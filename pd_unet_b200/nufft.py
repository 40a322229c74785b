"""Radial-MRI operators with the call shapes of torchkbnufft >= 1.0 ([RECALL], SURVEY.md section 8b;
the reference reaches the library through its unmounted MRI branch, /root/reference/README.md:3-5):

    KbNufft(im_size, grid_size=None, numpoints=6, n_shift=None, table_oversamp=2**10,
            kbwidth=2.34, order=0.0)(image, omega, interp_mats=None, smaps=None, norm=None)
    KbNufftAdjoint(...)(data, omega, interp_mats=None, smaps=None, norm=None)
    KbInterp(...)(image, omega) / KbInterpAdjoint(...)(data, omega)
    calc_density_compensation_function(ktraj, im_size, num_iterations=10, ...)
    calc_toeplitz_kernel(omega, im_size, weights=None, norm=None, ...) / ToepNufft()(image, kernel, smaps=None, norm=None)
    toep_cg(b, kernel, smaps=None, lam=0.0, x0=None, max_iter=10, tol=0.0): CG on (ToepNufft + lam I) x = b

image: complex64 [B, C, N0, N1]; omega: float32 [2, M] radians (or [B, 2, M]); data: complex64
[B, C, M].  With smaps [1 or B, coils, N0, N1] the forward expands a one-channel image to the
coils and the adjoint combines them.  Both directions are differentiable (each is the other's
conjugate transpose), in the maps too.  The modules register no parameters and no persistent buffers, so a model
containing them has the same state_dict as one without.

Everything numeric happens in libpdu_b200.so (pd_unet_b200/csrc/nufft.cu).  No CPU path.
"""
from __future__ import annotations

import ctypes as C
import math
from collections import OrderedDict
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch
from torch import nn

from ._lib import NUFFT_IMAGE_SPLIT, NUFFT_KDATA_SPLIT, PDU_EUNSUPPORTED, PduError, check, lib, require_cuda, stream_ptr


# ----------------------------------------------------------------------------- tables (host, float64)
def kaiser_bessel_table(n: int, k: int, numpoints: int, table_oversamp: int, kbwidth: float) -> np.ndarray:
    """complex128 [J L + 1]: kb(u) exp(-i (2 pi / K) ((N - 1) / 2) u) at u = q / L - J / 2
    (Fessler's NUFFT table, order 0)."""
    J, L = numpoints, table_oversamp
    u = np.arange(J * L + 1, dtype=np.float64) / L - J / 2.0
    inside = np.abs(u) < J / 2.0
    arg = np.sqrt(np.where(inside, 1.0 - (u / (J / 2.0)) ** 2, 0.0))
    alpha = kbwidth * J
    kb = np.where(inside, np.i0(alpha * arg) / np.i0(alpha), 0.0)
    return kb * np.exp(-1j * (2.0 * np.pi / k) * ((n - 1) / 2.0) * u)


def kaiser_bessel_scaling(n: int, k: int, numpoints: int, kbwidth: float) -> np.ndarray:
    """float64 [N]: reciprocal of the Kaiser-Bessel kernel's Fourier transform (apodisation correction)."""
    J = numpoints
    alpha = kbwidth * J
    om = (np.arange(n, dtype=np.float64) - (n - 1) / 2.0) / k
    w2 = alpha ** 2 - (np.pi * J * om) ** 2
    w = np.sqrt(np.abs(w2))
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(w2 > 0, np.sinh(w) / w, np.sin(w) / w)
    ratio = np.where(w == 0, 1.0, ratio)
    return np.i0(alpha) / (J * ratio)


# Device handles of plans collected while the current stream was capturing a CUDA graph.  Destroying a plan calls
# cufftDestroy and cudaFree, which invalidate a capture, and a collection can happen inside one: an MRI model refers to
# itself through its operator closures, so the cyclic garbage collector frees it (and its plans) at whatever allocation
# triggers a collection.  The handles are destroyed with the next plan collected outside a capture.
_DEFERRED_DESTROY: list = []


class _Plan:
    """Owns one pdu_nufft_plan_t per device."""

    def __init__(self, im_size, grid_size, numpoints, n_shift, table_oversamp, kbwidth, order):
        if len(im_size) != 2:
            raise NotImplementedError("only 2-D transforms are implemented (radial MRI slices)")
        if float(order) != 0.0:
            raise NotImplementedError("only order-0 Kaiser-Bessel kernels are implemented")
        self.im_size = tuple(int(v) for v in im_size)
        self.grid_size = tuple(int(v) for v in (grid_size or [2 * n for n in self.im_size]))
        self.n_shift = tuple(int(v) for v in (n_shift or [n // 2 for n in self.im_size]))
        self.numpoints = int(numpoints if np.isscalar(numpoints) else numpoints[0])
        self.table_oversamp = int(table_oversamp if np.isscalar(table_oversamp) else table_oversamp[0])
        self.kbwidth = float(kbwidth)
        self.tables = [kaiser_bessel_table(n, k, self.numpoints, self.table_oversamp, self.kbwidth).astype(np.complex64)
                       for n, k in zip(self.im_size, self.grid_size)]
        self.scaling = [kaiser_bessel_scaling(n, k, self.numpoints, self.kbwidth).astype(np.float32)
                        for n, k in zip(self.im_size, self.grid_size)]
        self._handles: Dict[int, C.c_void_p] = {}
        # per-trajectory precomputation (row bins of the fused path, CSR form of the adjoint interpolator), keyed by
        # the trajectory tensor's identity; a fixed trajectory is reused by every unrolled iteration / training step
        self._traj: "OrderedDict[tuple, dict]" = OrderedDict()
        self.traj_cache_bytes = 512 << 20
        # "auto": the gather where it is faster (measured on B200: >= 8 planes per call, see _csr_for; with fewer
        # planes the atomic scatter wins -- 67 vs 180 us at 256 spokes x 1 plane); True: always (bit-reproducible
        # adjoint); False: never.  Only the generic path (grids without a fused path, KbInterpAdjoint) looks at it.
        self.use_csr = "auto"
        # the fused path (csrc/nufft_fused.cu): True -- wherever the library has one for the grid; False -- never;
        # "auto" -- where it measured faster on B200 (tools/prof_nufft.py, profiles/r02_nufft_timings.txt): from 8 planes
        # per call up (below that a call is ~700 short-lived CTAs and the generic path's wide gathers win: 24 vs 36 us
        # at 256^2 x 1 plane), and for the adjoint only while the plane count is moderate (_bins_for: 64 planes of
        # 640^2 with coil maps: fused 294 us, generic sorted gather + register FFT 253 us; forward 206 vs 261 us)
        self.use_fused = "auto"
        self.fused_max_row = 4096     # "auto": no fused path for a trajectory whose heaviest grid row has more entries

    # -------------------------------------------------------------- per-trajectory cache
    def _entry(self, omega: torch.Tensor) -> dict:
        key = (omega.data_ptr(), omega._version, tuple(omega.shape), omega.device)
        ent = self._traj.get(key)
        if ent is None:
            ent = {"omega": omega, "bins": None, "csr": None, "events": []}   # omega kept alive: its address cannot be reused
            self._traj[key] = ent
        else:
            self._traj.move_to_end(key)
        return ent

    def _trim(self) -> None:
        def nbytes(e):
            return sum(t.numel() for t in (e["bins"], e["csr"]) if t is not None)
        while len(self._traj) > 1 and (len(self._traj) > 16 or sum(nbytes(e) for e in self._traj.values()) > self.traj_cache_bytes):
            self._traj.popitem(last=False)

    @staticmethod
    def _built(ent: dict) -> None:
        """Remember where the build ran so that a later use on another stream can wait for it."""
        ev = torch.cuda.Event()
        ev.record()
        ent["events"].append((torch.cuda.current_stream(), ev))

    @staticmethod
    def _wait(ent: dict) -> None:
        cur = torch.cuda.current_stream()
        if torch.cuda.is_current_stream_capturing():
            return                      # graph capture follows eager warm-up calls and a device synchronisation
        for st, ev in ent["events"]:
            if st != cur:
                cur.wait_event(ev)

    def _keep_prefix(self, buf: torch.Tensor, persist: int) -> torch.Tensor:
        """Only the head of a build buffer is needed afterwards; the sort scratch behind it (about two thirds) goes
        back to the allocator (stream-ordered, so the pending build kernels are safe)."""
        return buf[:persist].clone() if persist < buf.numel() else buf

    def _bins_for(self, omega: torch.Tensor, planes: int = 1 << 30, adjoint: bool = False, split: bool = False):
        """Row bins of the fused path for this trajectory (None when the generic path is to be used)."""
        L, h = lib(), self.handle(omega.device)
        if not self.use_fused or not L.pdu_nufft_has_fused_path(h):
            return None
        if self.use_fused == "auto":
            # measured policy (profiles/r02_nufft_timings.txt, profiles/r02_nufft_policy.txt): the row-binned kernels pay
            # per (sample, row) entry, so they win for sparse trajectories -- samples per grid cell rho <= 0.15
            # (configs[3]: 0.075) -- and lose by 2 - 8 x for dense ones (rho >= 0.5).  (While the generic adjoint still
            # scattered with atomics below 16 planes the fused one was also used up to rho = 0.3 there; against the
            # sorted gather from 8 planes it no longer pays: rho = 0.25, 8 / 12 planes, generic / fused us: 128^2
            # 48 / 60, 48 / 61; 256^2 91 / 110, 118 / 118; 512^2 294 / 253, 339 / 521.)
            rho = omega.shape[1] / float(self.grid_size[0] * self.grid_size[1])
            sparse = rho <= 0.15
            # adjoint: from a grid-dependent plane count on, the sorted gather (4 lanes per cell x 16 planes, non-empty cells
            # only, since r02) + FFT passes beat the row-binned kernel (tools/prof_nufft_adj_policy.py, REPS=21, generic /
            # fused us: 128^2 x 32 spokes 16 / 48 / 64 planes 44 / 65 / 71 against 38 / 63 / 77; 256^2 x 48 16 / 24 / 32 / 64
            # 71 / 85 / 101 / 173 against 65 / 91 / 114 / 208; 320^2 x 48 16 / 24 / 32 / 64 89 / 114 / 138 / 245 against
            # 85 / 116 / 146 / 273; 512^2 x 96 8 / 16 / 32 124 / 208 / 392 against 124 / 226 / 484; 1024^2 x 128 8 / 16
            # 419 / 744 against 484 / 1111)
            many = adjoint and planes >= {256: 64, 512: 24, 640: 32, 1024: 16}.get(self.grid_size[0], 8)
            if planes < 8 or not sparse or many:
                return None
        ent = self._entry(omega)
        if ent["bins"] is None:
            persist = C.c_size_t(0)
            nbytes = L.pdu_nufft_bins_bytes(h, omega.shape[1], C.byref(persist))
            buf = torch.empty(nbytes, dtype=torch.uint8, device=omega.device)
            check(L.pdu_nufft_bins_build(h, omega.data_ptr(), omega.shape[1], buf.data_ptr(), buf.numel(), stream_ptr()),
                  "pdu_nufft_bins_build")
            ent["bins"] = self._keep_prefix(buf, persist.value)
            self._built(ent)
            self._trim()
            # entries of the heaviest grid row (header word 7): one small read-back per trajectory, at build time
            ent["max_row"] = (int(ent["bins"][:64].cpu().view(torch.int32)[7])
                              if not torch.cuda.is_current_stream_capturing() else 0)
        else:
            self._wait(ent)
        if self.use_fused == "auto" and ent.get("max_row", 0) > self.fused_max_row:
            return None       # a few very heavy rows (dense or concentrated trajectory) serialise the row kernels
        return ent["bins"]

    def _csr_for(self, omega: torch.Tensor, planes: int = 1 << 30):
        """The sorted-gather form of the adjoint interpolator for this trajectory, built on first use."""
        # from 8 planes (16 before the gather went to 4 lanes per cell; tools/prof_nufft_csr_policy.py, atomics / sorted us:
        # 8 planes of 512^2 x 256 spokes 406 / 282, of 320^2 x 48 83 / 73, of 256^2 x 256 251 / 266; 4 planes 134 / 175)
        # -- where the plane-interleaved copy of the samples fits the call's scratch (M <= about three quarters of the grid cells); a denser
        # trajectory runs the planar form of the gather, which only pays from 16 planes (256^2 x 512 spokes, 8 planes:
        # 396 against 374 us for the scatter; 16 planes: 527 against 722)
        if self.use_csr == "auto":
            n0, n1 = self.im_size
            k0, k1 = self.grid_size
            fits = omega.shape[1] * ((planes + 3) & ~3) <= planes * (max(n0 * k1, k0 * n1) + n0 * n1)
            if planes < (8 if fits else 16):
                return None
        if self.use_csr is False:
            return None
        ent = self._entry(omega)
        if ent["csr"] is None:
            L, h = lib(), self.handle(omega.device)
            persist = C.c_size_t(0)
            nbytes = L.pdu_nufft_csr_bytes2(h, omega.shape[1], C.byref(persist))
            buf = torch.empty(nbytes, dtype=torch.uint8, device=omega.device)
            check(L.pdu_nufft_csr_build(h, omega.data_ptr(), omega.shape[1], buf.data_ptr(), buf.numel(), stream_ptr()),
                  "pdu_nufft_csr_build")
            ent["csr"] = self._keep_prefix(buf, persist.value)
            self._built(ent)
            self._trim()
        else:
            self._wait(ent)
        return ent["csr"]

    def handle(self, device: torch.device) -> C.c_void_p:
        idx = device.index if device.index is not None else torch.cuda.current_device()
        h = self._handles.get(idx)
        if h is None:
            h = C.c_void_p()
            t0, t1 = (np.ascontiguousarray(t) for t in self.tables)
            s0, s1 = (np.ascontiguousarray(s) for s in self.scaling)
            with torch.cuda.device(idx):
                check(lib().pdu_nufft_plan_create(C.byref(h), self.im_size[0], self.im_size[1], self.grid_size[0],
                                                  self.grid_size[1], self.numpoints, self.table_oversamp,
                                                  self.n_shift[0], self.n_shift[1], t0.ctypes.data, t1.ctypes.data,
                                                  s0.ctypes.data, s1.ctypes.data), "pdu_nufft_plan_create")
            self._handles[idx] = h
        return h

    def __deepcopy__(self, memo):  # noqa: D105
        # device handles are per-process resources: a copy starts without any and re-creates them lazily
        return _Plan(self.im_size, self.grid_size, self.numpoints, self.n_shift, self.table_oversamp, self.kbwidth, 0.0)

    def __getstate__(self):
        raise TypeError("a NUFFT plan holds device handles and cannot be pickled; rebuild the module instead")

    def __del__(self):
        try:
            if not self._handles:
                return
            _DEFERRED_DESTROY.extend(self._handles.values())
            if torch.cuda.is_current_stream_capturing():
                return
            while _DEFERRED_DESTROY:
                lib().pdu_nufft_plan_destroy(_DEFERRED_DESTROY.pop())
        except Exception:
            pass

    def scale(self, norm: Optional[str]) -> float:
        if norm is None:
            return 1.0
        if norm == "ortho":
            return 1.0 / math.sqrt(self.grid_size[0] * self.grid_size[1])
        raise ValueError("norm must be None or 'ortho'")

    # -------------------------------------------------------------- C-ABI calls (single trajectory)
    def _omega(self, omega: torch.Tensor) -> torch.Tensor:
        omega = require_cuda(omega, torch.float32, "omega")
        if omega.dim() != 2 or omega.shape[0] != 2:
            raise ValueError(f"omega must be [2, M], got {tuple(omega.shape)}")
        return omega

    def _smaps(self, smaps, batch):
        if smaps is None:
            return None, 0, 1
        smaps = require_cuda(smaps, torch.complex64, "smaps")
        if smaps.dim() == 3:
            smaps = smaps[None]
        if smaps.dim() != 4 or tuple(smaps.shape[-2:]) != self.im_size or smaps.shape[0] not in (1, batch):
            raise ValueError(f"smaps must be [1 or {batch}, coils, {self.im_size[0]}, {self.im_size[1]}]")
        return smaps, smaps.shape[1], smaps.shape[0]

    # Layouts.  split=False: complex64 tensors, image [B, C, N0, N1], data [B, C, M] (torchkbnufft's).
    # split=True: float32 tensors with the real and imaginary parts as neighbouring channels, image [B, 2 C, N0, N1],
    # data [B, 2 C, M] -- what PD-UNet's CNN blocks carry, so the model needs no permute / view_as_complex passes.
    @staticmethod
    def _split_to_complex(x: torch.Tensor, weight: Optional[torch.Tensor] = None) -> torch.Tensor:
        """[B, 2 C, *s] float32 -> [B, C, *s] complex64 (x weight[*s]), one pass of the library's layout kernel."""
        B, C2 = x.shape[:2]
        out = torch.empty((B, C2 // 2) + tuple(x.shape[2:]), dtype=torch.complex64, device=x.device)
        n = out[0, 0].numel()
        if out.numel():
            check(lib().pdu_complex_from_split_f32(x.data_ptr(), out.data_ptr(), weight.data_ptr() if weight is not None else None,
                                                   B * (C2 // 2), n, stream_ptr()), "pdu_complex_from_split_f32")
        return out

    @staticmethod
    def _complex_to_split(z: torch.Tensor) -> torch.Tensor:
        B, Cc = z.shape[:2]
        out = torch.empty((B, 2 * Cc) + tuple(z.shape[2:]), dtype=torch.float32, device=z.device)
        if out.numel():
            check(lib().pdu_split_from_complex_f32(z.data_ptr(), out.data_ptr(), B * Cc, z[0, 0].numel(), stream_ptr()),
                  "pdu_split_from_complex_f32")
        return out

    def _chunks(self, L, h, B: int, coils: int, M: int):
        """Batch chunks that keep the fused path's scratch under 1 GiB."""
        per = max(1, L.pdu_nufft_binned_workspace_bytes(h, coils, M))
        cb = max(1, min(B, (1 << 30) // per))
        return [(b0, min(B, b0 + cb)) for b0 in range(0, B, cb)]

    def forward(self, image, omega, smaps, norm, split: bool = False):
        image = require_cuda(image, torch.float32 if split else torch.complex64, "image")
        if image.dim() != 4 or tuple(image.shape[-2:]) != self.im_size or (split and image.shape[1] % 2):
            raise ValueError(f"image must be [B, C, {self.im_size[0]}, {self.im_size[1]}], got {tuple(image.shape)}")
        omega = self._omega(omega)
        B, M = image.shape[0], omega.shape[1]
        ci = image.shape[1] // 2 if split else image.shape[1]
        smaps, coils, sb = self._smaps(smaps, B)
        if smaps is None:
            coils = ci
        elif ci != 1:
            raise ValueError("with smaps the image must have one channel")
        out = (torch.empty((B, 2 * coils, M), dtype=torch.float32, device=image.device) if split else
               torch.empty((B, coils, M), dtype=torch.complex64, device=image.device))
        if B == 0 or M == 0:
            return out
        with torch.cuda.device(image.device):
            L, h = lib(), self.handle(image.device)
            bins = self._bins_for(omega, B * coils, split=split)
            if bins is not None:
                flags = (NUFFT_IMAGE_SPLIT | NUFFT_KDATA_SPLIT) if split else 0
                for b0, b1 in self._chunks(L, h, B, coils, M):
                    nb = b1 - b0
                    ws = torch.empty(L.pdu_nufft_binned_workspace_bytes(h, nb * coils, M), dtype=torch.uint8, device=image.device)
                    sm = None if smaps is None else (smaps if sb == 1 else smaps[b0:b1])
                    check(L.pdu_nufft_fwd_binned_c64(h, image[b0:b1].data_ptr(), out[b0:b1].data_ptr(),
                                                     sm.data_ptr() if sm is not None else None, nb, coils, 1 if sb == 1 else nb, M,
                                                     self.scale(norm), bins.data_ptr(), flags, ws.data_ptr(), ws.numel(),
                                                     stream_ptr()), "pdu_nufft_fwd_binned_c64")
                return out
            if split:
                return self._complex_to_split(self.forward(self._split_to_complex(image), omega, smaps, norm))
            ws = torch.empty(L.pdu_nufft_workspace_bytes(h, B * coils), dtype=torch.uint8, device=image.device)
            check(L.pdu_nufft_fwd_c64(h, image.data_ptr(), out.data_ptr(), omega.data_ptr(),
                                      smaps.data_ptr() if smaps is not None else None, B, coils, sb, M,
                                      self.scale(norm), ws.data_ptr(), ws.numel(), stream_ptr()), "pdu_nufft_fwd_c64")
        return out

    def adjoint(self, data, omega, smaps, norm, split: bool = False, kweight: Optional[torch.Tensor] = None):
        """kweight: float32 [M] multiplied into the samples first (density compensation)."""
        data = require_cuda(data, torch.float32 if split else torch.complex64, "data")
        omega = self._omega(omega)
        if data.dim() != 3 or data.shape[-1] != omega.shape[1] or (split and data.shape[1] % 2):
            raise ValueError(f"data must be [B, C, {omega.shape[1]}], got {tuple(data.shape)}")
        B, M = data.shape[0], data.shape[2]
        coils = data.shape[1] // 2 if split else data.shape[1]
        smaps, sc, sb = self._smaps(smaps, B)
        if smaps is not None and sc != coils:
            raise ValueError(f"data has {coils} coils, smaps {sc}")
        if kweight is not None:
            kweight = require_cuda(kweight, torch.float32, "kweight").reshape(-1)
            if kweight.numel() != M:
                raise ValueError(f"kweight must have {M} entries")
        co = 1 if smaps is not None else coils
        out = (torch.empty((B, 2 * co) + self.im_size, dtype=torch.float32, device=data.device) if split else
               torch.empty((B, co) + self.im_size, dtype=torch.complex64, device=data.device))
        if B == 0:
            return out
        if M == 0:
            return out.zero_()
        with torch.cuda.device(data.device):
            L, h = lib(), self.handle(data.device)
            bins = self._bins_for(omega, B * coils, adjoint=True, split=split)
            if bins is not None:
                flags = (NUFFT_IMAGE_SPLIT | NUFFT_KDATA_SPLIT) if split else 0
                for b0, b1 in self._chunks(L, h, B, coils, M):
                    nb = b1 - b0
                    ws = torch.empty(L.pdu_nufft_binned_workspace_bytes(h, nb * coils, M), dtype=torch.uint8, device=data.device)
                    sm = None if smaps is None else (smaps if sb == 1 else smaps[b0:b1])
                    check(L.pdu_nufft_adj_binned_c64(h, data[b0:b1].data_ptr(), out[b0:b1].data_ptr(),
                                                     sm.data_ptr() if sm is not None else None,
                                                     kweight.data_ptr() if kweight is not None else None, nb, coils,
                                                     1 if sb == 1 else nb, M, self.scale(norm), bins.data_ptr(), flags,
                                                     ws.data_ptr(), ws.numel(), stream_ptr()), "pdu_nufft_adj_binned_c64")
                return out
            if split:            # generic path: the library's layout kernels around the complex64 entry points
                return self._complex_to_split(self.adjoint(self._split_to_complex(data, kweight), omega, smaps, norm))
            if kweight is not None:
                return self.adjoint(data * kweight, omega, smaps, norm)
            ws = torch.empty(L.pdu_nufft_workspace_bytes(h, B * coils), dtype=torch.uint8, device=data.device)
            csr = self._csr_for(omega, B * coils)
            check(L.pdu_nufft_adj_csr_c64(h, data.data_ptr(), out.data_ptr(), omega.data_ptr(),
                                          smaps.data_ptr() if smaps is not None else None, B, coils, sb, M,
                                          self.scale(norm), csr.data_ptr() if csr is not None else None, ws.data_ptr(),
                                          ws.numel(), stream_ptr()), "pdu_nufft_adj_c64")
        return out

    def smaps_grad(self, data, omega, q, gs, norm, split: bool = False, kweight: Optional[torch.Tensor] = None,
                   accumulate: bool = False) -> None:
        """gs [1 or B, coils, N0, N1] (+)= sum over b of the un-combined adjoint of data[b] (as adjoint() would run it)
        times conj(q[b]); q is the image side [B, 1, N0, N1] (split: [B, 2, N0, N1] float32).  A shared map (gs[0])
        sums the batch in increasing order, carried from chunk to chunk."""
        omega = self._omega(omega)
        data, q = data.contiguous(), q.contiguous()
        if kweight is not None:
            kweight = require_cuda(kweight, torch.float32, "kweight").reshape(-1)
        B, M = data.shape[0], data.shape[2]
        coils = data.shape[1] // 2 if split else data.shape[1]
        per_batch = gs.shape[0] != 1
        if B == 0 or M == 0:
            if not accumulate:
                gs.zero_()
            return
        L, h = lib(), self.handle(data.device)
        bins = self._bins_for(omega, B * coils, adjoint=True, split=split)
        if bins is not None:
            flags = (NUFFT_IMAGE_SPLIT | NUFFT_KDATA_SPLIT) if split else 0
            for b0, b1 in self._chunks(L, h, B, coils, M):
                nb = b1 - b0
                ws = torch.empty(L.pdu_nufft_binned_workspace_bytes(h, nb * coils, M), dtype=torch.uint8, device=data.device)
                g = gs[b0:b1] if per_batch else gs
                check(L.pdu_nufft_adj_smaps_grad_c64(h, data[b0:b1].data_ptr(), q[b0:b1].data_ptr(), g.data_ptr(), None, None,
                                                     bins.data_ptr(), kweight.data_ptr() if kweight is not None else None, nb,
                                                     coils, g.shape[0], M, self.scale(norm), flags,
                                                     1 if (accumulate or (b0 > 0 and not per_batch)) else 0, ws.data_ptr(),
                                                     ws.numel(), stream_ptr()), "pdu_nufft_adj_smaps_grad_c64")
            return
        # generic path: complex64 kdata with the weights applied, as adjoint() feeds pdu_nufft_adj_csr_c64
        if split:
            data = self._split_to_complex(data, kweight)
        elif kweight is not None:
            data = data * kweight
        ws = torch.empty(L.pdu_nufft_workspace_bytes(h, B * coils), dtype=torch.uint8, device=data.device)
        csr = self._csr_for(omega, B * coils)
        check(L.pdu_nufft_adj_smaps_grad_c64(h, data.data_ptr(), q.data_ptr(), gs.data_ptr(), omega.data_ptr(),
                                             csr.data_ptr() if csr is not None else None, None, None, B, coils, gs.shape[0], M,
                                             self.scale(norm), NUFFT_IMAGE_SPLIT if split else 0, 1 if accumulate else 0,
                                             ws.data_ptr(), ws.numel(), stream_ptr()), "pdu_nufft_adj_smaps_grad_c64")

    def interp(self, grid, omega):
        grid = require_cuda(grid, torch.complex64, "grid")
        if grid.dim() != 4 or tuple(grid.shape[-2:]) != self.grid_size:
            raise ValueError(f"grid must be [B, C, {self.grid_size[0]}, {self.grid_size[1]}]")
        omega = self._omega(omega)
        B, Cc, M = grid.shape[0], grid.shape[1], omega.shape[1]
        out = torch.empty((B, Cc, M), dtype=torch.complex64, device=grid.device)
        if B * Cc == 0 or M == 0:
            return out
        with torch.cuda.device(grid.device):
            check(lib().pdu_nufft_interp_fwd_c64(self.handle(grid.device), grid.data_ptr(), out.data_ptr(),
                                                 omega.data_ptr(), B * Cc, M, stream_ptr()), "pdu_nufft_interp_fwd_c64")
        return out

    def interp_adjoint(self, data, omega):
        data = require_cuda(data, torch.complex64, "data")
        omega = self._omega(omega)
        if data.dim() != 3 or data.shape[-1] != omega.shape[1]:
            raise ValueError(f"data must be [B, C, {omega.shape[1]}]")
        B, Cc, M = data.shape
        if B * Cc == 0 or M == 0:
            return torch.zeros((B, Cc) + self.grid_size, dtype=torch.complex64, device=data.device)
        with torch.cuda.device(data.device):
            csr = self._csr_for(omega, B * Cc)
            if csr is not None:      # the gather writes every cell
                out = torch.empty((B, Cc) + self.grid_size, dtype=torch.complex64, device=data.device)
                check(lib().pdu_nufft_interp_adj_csr_c64(self.handle(data.device), data.data_ptr(), out.data_ptr(),
                                                         csr.data_ptr(), B * Cc, M, stream_ptr()),
                      "pdu_nufft_interp_adj_csr_c64")
            else:                    # the scatter accumulates
                out = torch.zeros((B, Cc) + self.grid_size, dtype=torch.complex64, device=data.device)
                check(lib().pdu_nufft_interp_adj_c64(self.handle(data.device), data.data_ptr(), out.data_ptr(),
                                                     omega.data_ptr(), B * Cc, M, stream_ptr()), "pdu_nufft_interp_adj_c64")
        return out


def _per_trajectory(fn, x, omega, smaps, *rest):
    """torchkbnufft lets omega carry a batch axis ([B, 2, M]); each trajectory is its own call."""
    if omega.dim() == 2:
        return fn(x, omega, smaps, *rest)
    if omega.dim() != 3 or omega.shape[0] != x.shape[0]:
        raise ValueError("batched omega must be [B, 2, M] with the batch of the data")
    outs = []
    for b in range(x.shape[0]):
        sm = None if smaps is None else (smaps if smaps.shape[0] == 1 else smaps[b:b + 1])
        outs.append(fn(x[b:b + 1], omega[b], sm, *rest))
    return torch.cat(outs, dim=0)


def _nufft_smaps_grad(plan: _Plan, data, omega, q, smaps, norm, split, kweight) -> torch.Tensor:
    """The coil-map gradient sum_b A^H(w data[b, c]) conj(q[b]) in the shape of smaps (3-D or 4-D); a batched omega runs
    per trajectory, a shared map summing the batch in increasing order."""
    sm = smaps if smaps.dim() == 4 else smaps[None]
    gs = torch.empty(sm.shape, dtype=torch.complex64, device=data.device)
    with torch.cuda.device(data.device):
        if omega.dim() == 2:
            plan.smaps_grad(data, omega, q, gs, norm, split, kweight)
        else:
            for b in range(data.shape[0]):
                plan.smaps_grad(data[b:b + 1], omega[b], q[b:b + 1], gs if gs.shape[0] == 1 else gs[b:b + 1], norm, split,
                                kweight, accumulate=gs.shape[0] == 1 and b > 0)
    return gs.reshape(smaps.shape)


class _NufftFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, omega, smaps, plan, norm, adjoint, split=False, kweight=None):
        ctx.plan, ctx.norm, ctx.adjoint, ctx.split, ctx.kweight = plan, norm, adjoint, split, kweight
        if smaps is None:
            ctx.save_for_backward(omega)
        elif ctx.needs_input_grad[2]:        # the map gradient pairs the input with the incoming gradient
            ctx.save_for_backward(omega, smaps, x)
        else:
            ctx.save_for_backward(omega, smaps)
        if adjoint:
            return _per_trajectory(plan.adjoint, x, omega, smaps, norm, split, kweight)
        return _per_trajectory(plan.forward, x, omega, smaps, norm, split)

    @staticmethod
    def backward(ctx, grad):
        saved = ctx.saved_tensors
        omega, smaps = saved[0], (saved[1] if len(saved) > 1 else None)
        grad = grad.contiguous()
        g = gs = None
        if ctx.needs_input_grad[0] or not ctx.needs_input_grad[2]:
            if ctx.adjoint:       # x = A^H (w y)  =>  dy = w A dx
                g = _per_trajectory(ctx.plan.forward, grad, omega, smaps, ctx.norm, ctx.split)
                if ctx.kweight is not None:
                    g = g * ctx.kweight.reshape(-1)
            else:
                g = _per_trajectory(ctx.plan.adjoint, grad, omega, smaps, ctx.norm, ctx.split)
        if smaps is not None and ctx.needs_input_grad[2]:
            x = saved[2]
            # forward  y[b, c] = A(S_c x_b):              gS_c = sum_b A^H(g[b, c]) conj(x_b)
            # adjoint  x_b = sum_c conj(S_c) A^H(w y[b, c]):  gS_c = sum_b A^H(w y[b, c]) conj(g_b)
            if ctx.adjoint:
                gs = _nufft_smaps_grad(ctx.plan, x, omega, grad, smaps, ctx.norm, ctx.split, ctx.kweight)
            else:
                gs = _nufft_smaps_grad(ctx.plan, grad, omega, x, smaps, ctx.norm, ctx.split, None)
        return g, None, gs, None, None, None, None, None


class _InterpFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, omega, plan, adjoint):
        ctx.plan, ctx.adjoint = plan, adjoint
        ctx.save_for_backward(omega)
        fn = plan.interp_adjoint if adjoint else plan.interp
        return _per_trajectory(lambda a, o, s: fn(a, o), x, omega, None)

    @staticmethod
    def backward(ctx, grad):
        (omega,) = ctx.saved_tensors
        fn = ctx.plan.interp if ctx.adjoint else ctx.plan.interp_adjoint
        return _per_trajectory(lambda a, o, s: fn(a, o), grad.contiguous(), omega, None), None, None, None


class _KbModule(nn.Module):
    def __init__(self, im_size: Sequence[int], grid_size: Optional[Sequence[int]] = None, numpoints=6,
                 n_shift: Optional[Sequence[int]] = None, table_oversamp=2 ** 10, kbwidth: float = 2.34,
                 order=0.0, dtype=None, device=None):
        super().__init__()
        order0 = float(order if np.isscalar(order) else order[0])
        self._plan = _Plan(im_size, grid_size, numpoints, n_shift, table_oversamp, kbwidth, order0)
        self.im_size, self.grid_size, self.n_shift = self._plan.im_size, self._plan.grid_size, self._plan.n_shift
        self.numpoints, self.table_oversamp = self._plan.numpoints, self._plan.table_oversamp

    @staticmethod
    def _no_interp_mats(interp_mats):
        if interp_mats is not None:
            raise NotImplementedError("sparse-matrix interpolation is not implemented; pass interp_mats=None "
                                      "(table interpolation, torchkbnufft's default)")


class KbNufft(_KbModule):
    """image [B, C, N0, N1] -> k-space samples [B, C (or coils), M].  [RECALL] torchkbnufft.KbNufft.

    Differentiable in the image and in smaps: grad_S[c] = sum_b A^H(g[b, c]) conj(x_b) over the batch elements sharing
    a map, one adjoint launch set ending in the library's map-gradient kernel; maps that need no gradient cost
    nothing extra."""

    def forward(self, image, omega, interp_mats=None, smaps=None, norm: Optional[str] = None, split: bool = False):
        """split=True (an extension): image float32 [B, 2 C, N0, N1] with (re, im) as neighbouring channels ->
        float32 [B, 2 coils, M]; no complex tensors, no layout passes around the operator."""
        self._no_interp_mats(interp_mats)
        return _NufftFn.apply(image, omega, smaps, self._plan, norm, False, split)


class KbNufftAdjoint(_KbModule):
    """samples [B, C, M] -> image [B, C (or 1), N0, N1].  [RECALL] torchkbnufft.KbNufftAdjoint.

    Differentiable in the samples and in smaps: grad_S[c] = sum_b A^H(kweight y[b, c]) conj(g_b) over the batch
    elements sharing a map (the un-combined adjoint of the input, reduced by the library's map-gradient kernel)."""

    def forward(self, data, omega, interp_mats=None, smaps=None, norm: Optional[str] = None, split: bool = False,
                kweight: Optional[torch.Tensor] = None):
        """Extensions: split=True as in KbNufft; kweight float32 [M] is multiplied into the samples on load (the
        density compensation that otherwise is a separate pass over the data)."""
        self._no_interp_mats(interp_mats)
        return _NufftFn.apply(data, omega, smaps, self._plan, norm, True, split, kweight)


class KbInterp(_KbModule):
    """oversampled Cartesian k-space [B, C, K0, K1] -> samples [B, C, M].  [RECALL] torchkbnufft.KbInterp."""

    def forward(self, image, omega, interp_mats=None):
        self._no_interp_mats(interp_mats)
        return _InterpFn.apply(image, omega, self._plan, False)


class KbInterpAdjoint(_KbModule):
    """samples [B, C, M] -> gridded k-space [B, C, K0, K1].  [RECALL] torchkbnufft.KbInterpAdjoint."""

    def forward(self, data, omega, interp_mats=None):
        self._no_interp_mats(interp_mats)
        return _InterpFn.apply(data, omega, self._plan, True)


def calc_density_compensation_function(ktraj: torch.Tensor, im_size: Sequence[int], num_iterations: int = 10,
                                       grid_size: Optional[Sequence[int]] = None, numpoints=6,
                                       n_shift: Optional[Sequence[int]] = None, table_oversamp=2 ** 10,
                                       kbwidth: float = 2.34, order=0.0) -> torch.Tensor:
    """Pipe & Menon's iteration w <- w / |G G^H w| with the table interpolator only.
    [RECALL] torchkbnufft.calc_density_compensation_function; returns complex64 [1, 1, M]."""
    plan = _Plan(im_size, grid_size, numpoints, n_shift, table_oversamp, kbwidth, order)
    omega = require_cuda(ktraj, torch.float32, "ktraj")
    w = torch.ones((1, 1, omega.shape[1]), dtype=torch.complex64, device=omega.device)
    for _ in range(num_iterations):
        new = plan.interp(plan.interp_adjoint(w, omega), omega)
        w = w / new.abs()
    return w


# ----------------------------------------------------------------------------- Toeplitz-embedded normal operator
class _ToepPlan:
    """Owns one Toeplitz pdu_nufft_plan_t (grid 2 N, unit apodisation, no tables) per device for one image size."""

    def __init__(self, im_size: Tuple[int, int]):
        self.im_size = im_size
        self._handles: Dict[int, C.c_void_p] = {}

    def handle(self, device: torch.device) -> C.c_void_p:
        idx = device.index if device.index is not None else torch.cuda.current_device()
        h = self._handles.get(idx)
        if h is None:
            h = C.c_void_p()
            with torch.cuda.device(idx):
                rc = lib().pdu_toep_plan_create(C.byref(h), self.im_size[0], self.im_size[1])
            if rc == PDU_EUNSUPPORTED:
                raise NotImplementedError(f"no Toeplitz path for a {self.im_size[0]} x {self.im_size[1]} image (the 2 N "
                                          "embedding grid must factor into 2, 3, 5); there is no CPU fallback")
            check(rc, "pdu_toep_plan_create")
            self._handles[idx] = h
        return h

    def workspace_bytes(self, h, batch: int, coils: int) -> int:
        """Scratch of one batch chunk: the arithmetic of csrc/nufft.cu::tz_batch_chunk (512 MB, 65535 planes)."""
        L = lib()
        per = int(L.pdu_toep_workspace_bytes(h, 1))
        cb = min(batch, max(1, min((512 << 20) // per, 65535) // coils))
        return int(L.pdu_toep_workspace_bytes(h, cb * coils))

    def __del__(self):
        # the same deferred destruction as _Plan: a collection during a CUDA-graph capture must not free device memory
        try:
            if not self._handles:
                return
            _DEFERRED_DESTROY.extend(self._handles.values())
            if torch.cuda.is_current_stream_capturing():
                return
            while _DEFERRED_DESTROY:
                lib().pdu_nufft_plan_destroy(_DEFERRED_DESTROY.pop())
        except Exception:
            pass


_TOEP_PLANS: Dict[Tuple[int, int], _ToepPlan] = {}


def _toep_plan(im_size) -> _ToepPlan:
    key = tuple(int(v) for v in im_size)
    if len(key) != 2:
        raise NotImplementedError("only 2-D Toeplitz operators are implemented (radial MRI slices)")
    tp = _TOEP_PLANS.get(key)
    if tp is None:
        tp = _TOEP_PLANS[key] = _ToepPlan(key)
    return tp


def _check_norm(norm: Optional[str]) -> None:
    if norm not in (None, "ortho"):
        raise ValueError("norm must be None or 'ortho'")


def _toep_args(image: torch.Tensor, kernel: torch.Tensor, smaps: Optional[torch.Tensor], name: str = "image"):
    """Checked operands of a Toeplitz call: (image, kernel [1 or B, 2 N0, 2 N1], smaps or None, coils, smaps batch)."""
    image = require_cuda(image, torch.complex64, name)
    kernel = require_cuda(kernel, torch.complex64, "kernel")
    if image.dim() != 4:
        raise ValueError(f"{name} must be [B, C, N0, N1], got {tuple(image.shape)}")
    B, ci, N0, N1 = image.shape
    if kernel.dim() == 2:
        kernel = kernel[None]
    if kernel.dim() != 3 or tuple(kernel.shape[1:]) != (2 * N0, 2 * N1) or kernel.shape[0] not in (1, B):
        raise ValueError(f"kernel must be [2 N0, 2 N1] = [{2 * N0}, {2 * N1}] or [1 or {B}, {2 * N0}, {2 * N1}] for this image, "
                         f"got {tuple(kernel.shape)}")
    coils, sb = ci, 1
    if smaps is not None:
        smaps = require_cuda(smaps, torch.complex64, "smaps")
        if smaps.dim() == 3:
            smaps = smaps[None]
        if smaps.dim() != 4 or tuple(smaps.shape[-2:]) != (N0, N1) or smaps.shape[0] not in (1, B):
            raise ValueError(f"smaps must be [1 or {B}, coils, {N0}, {N1}]")
        if ci != 1:
            raise ValueError(f"with smaps the {name} must have one channel")
        coils, sb = smaps.shape[1], smaps.shape[0]
    return image, kernel, smaps, coils, sb


def _toep_apply(image: torch.Tensor, kernel: torch.Tensor, smaps: Optional[torch.Tensor], conj: bool) -> torch.Tensor:
    image, kernel, smaps, coils, sb = _toep_args(image, kernel, smaps)
    B, _, N0, N1 = image.shape
    out = torch.empty_like(image)
    if out.numel() == 0:
        return out
    with torch.cuda.device(image.device):
        tp = _toep_plan((N0, N1))
        h = tp.handle(image.device)
        L = lib()
        ws = torch.empty(tp.workspace_bytes(h, B, coils), dtype=torch.uint8, device=image.device)
        check(L.pdu_toep_apply_c64(h, image.data_ptr(), out.data_ptr(), kernel.data_ptr(), kernel.shape[0],
                                   smaps.data_ptr() if smaps is not None else None, B, coils, sb, 1 if conj else 0,
                                   ws.data_ptr(), ws.numel(), stream_ptr()), "pdu_toep_apply_c64")
    return out


def _toep_smaps_grad(x: torch.Tensor, g: torch.Tensor, kernel: torch.Tensor, smaps: torch.Tensor, out_scale: float) -> torch.Tensor:
    """out_scale * sum_b [T(S_c x_b) conj(g_b) + T^H(S_c g_b) conj(x_b)], the coil-map gradient of ToepNufft at (x, g), in
    the shape of smaps."""
    x, kernel, sm, coils, sb = _toep_args(x, kernel, smaps)
    g = require_cuda(g, torch.complex64, "grad").contiguous()
    B, _, N0, N1 = x.shape
    gs = torch.empty(sm.shape, dtype=torch.complex64, device=x.device)
    if B == 0:
        return gs.zero_().reshape(smaps.shape)
    with torch.cuda.device(x.device):
        tp = _toep_plan((N0, N1))
        h = tp.handle(x.device)
        ws = torch.empty(tp.workspace_bytes(h, B, coils), dtype=torch.uint8, device=x.device)
        check(lib().pdu_toep_smaps_grad_c64(h, x.data_ptr(), g.data_ptr(), gs.data_ptr(), kernel.data_ptr(), kernel.shape[0],
                                            sm.data_ptr(), B, coils, sb, 0, out_scale, 0, ws.data_ptr(), ws.numel(),
                                            stream_ptr()), "pdu_toep_smaps_grad_c64")
    return gs.reshape(smaps.shape)


class _ToepFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, kernel, smaps):
        if smaps is None:
            ctx.save_for_backward(kernel)
        elif ctx.needs_input_grad[2]:
            ctx.save_for_backward(kernel, smaps, x)
        else:
            ctx.save_for_backward(kernel, smaps)
        return _toep_apply(x, kernel, smaps, False)

    @staticmethod
    def backward(ctx, grad):
        saved = ctx.saved_tensors
        kernel, smaps = saved[0], (saved[1] if len(saved) > 1 else None)
        grad = grad.contiguous()
        gx = gs = None
        if ctx.needs_input_grad[0] or not ctx.needs_input_grad[2]:
            # T = P^T F^-1 diag(k) F P (with coil maps: sum_c S_c^H T S_c), so T^H is the same apply with conj(k): exact
            # for any complex kernel
            gx = _toep_apply(grad, kernel, smaps, True)
        if smaps is not None and ctx.needs_input_grad[2]:
            gs = _toep_smaps_grad(saved[2], grad, kernel, smaps, 1.0)
        return gx, None, gs


class ToepNufft(nn.Module):
    """The NUFFT normal operator A^H W A by Toeplitz embedding.  [RECALL] torchkbnufft.ToepNufft.

    forward(image, kernel, smaps=None, norm=None): image complex64 [B, C, N0, N1]; kernel complex64 [2 N0, 2 N1] or
    [1 or B, 2 N0, 2 N1] from calc_toeplitz_kernel.  Returns ifft2(kernel * fft2(zero_pad(x)))[..., :N0, :N1] for every
    channel, or with smaps [1 or B, coils, N0, N1] (image [B, 1, N0, N1]) sum_c conj(S_c) T(S_c x).  No interpolation:
    the cost does not depend on the trajectory length.

    norm is accepted with torchkbnufft's values and does not change the result [RECALL]: the FFT pair's normalisations
    multiply to the same total either way, and the NUFFT's scaling lives in the kernel (calc_toeplitz_kernel(norm=...)).
    Differentiable in the image (the backward is the same apply with the conjugate kernel, exact for any complex
    kernel) and in smaps: grad_S[c] = sum_b [T(S_c x_b) conj(g_b) + T^H(S_c g_b) conj(x_b)], two apply launch sets
    whose last pass walks the batch instead of the coils.  No gradient flows to the kernel.  No parameters, no
    buffers."""

    def forward(self, image, kernel, smaps=None, norm: Optional[str] = None):
        _check_norm(norm)
        return _ToepFn.apply(image, kernel, smaps)


def calc_toeplitz_kernel(omega: torch.Tensor, im_size: Sequence[int], weights: Optional[torch.Tensor] = None,
                         norm: Optional[str] = None, grid_size: Optional[Sequence[int]] = None, numpoints=6,
                         n_shift: Optional[Sequence[int]] = None, table_oversamp=2 ** 10, kbwidth: float = 2.34,
                         order=0.0) -> torch.Tensor:
    """The Toeplitz kernel of A^H W A for trajectory omega [2, M] (or [B, 2, M]: one kernel per trajectory).
    [RECALL] torchkbnufft.calc_toeplitz_kernel; returns complex64 [2 N0, 2 N1] (or [B, 2 N0, 2 N1]).

    kernel = fft2(p_circ), p[r] = s * sum_m w_m exp(i omega_m . r) for |r| < N in circulant layout; the point-spread
    function comes from two adjoint NUFFTs of the weights (omega, and omega with its first row negated) at the user's
    grid_size / numpoints / table, so it carries their Kaiser-Bessel approximation error.  s = 1 / (K0 K1) of the NUFFT
    grid for norm="ortho", 1 for None.  weights: real, float32 [M] / [1, 1, M] (or [B, 1, M] for a batched omega), or
    complex64 with a zero imaginary part (what calc_density_compensation_function returns); None means all ones.
    n_shift is accepted and ignored: the normal operator does not depend on it."""
    del n_shift
    _check_norm(norm)
    im_size = tuple(int(v) for v in im_size)
    tp = _toep_plan(im_size)
    omega = require_cuda(omega, torch.float32, "omega")
    h = tp.handle(omega.device)               # an unsupported size fails here, before any NUFFT work
    om = omega if omega.dim() == 3 else omega[None]
    if om.dim() != 3 or om.shape[1] != 2:
        raise ValueError(f"omega must be [2, M] or [B, 2, M], got {tuple(omega.shape)}")
    nk, M = om.shape[0], om.shape[2]
    if weights is None:
        w = torch.ones((nk, 1, M), dtype=torch.float32, device=omega.device)
    else:
        if not isinstance(weights, torch.Tensor) or not weights.is_cuda:
            raise PduError("weights must be a CUDA tensor (no CPU fallback)")
        if weights.is_complex():
            if bool((weights.imag != 0).any()):        # one read-back per kernel build
                raise ValueError("weights must be real: the kernel's Hermitian assembly assumes p(-r) = conj p(r)")
            weights = weights.real
        w = weights.to(torch.float32)
        if w.numel() == M:
            w = w.reshape(1, 1, M).expand(nk, 1, M)
        elif w.numel() == nk * M:
            w = w.reshape(nk, 1, M)
        else:
            raise ValueError(f"weights must have {M} entries (or {nk} x {M} for a batched omega), got {tuple(weights.shape)}")
    w = torch.complex(w, torch.zeros_like(w)).contiguous()
    plan = _Plan(im_size, grid_size, numpoints, (0, 0), table_oversamp, kbwidth, float(order if np.isscalar(order) else order[0]))
    scale = 1.0 / (plan.grid_size[0] * plan.grid_size[1]) if norm == "ortho" else 1.0
    flip = torch.tensor([-1.0, 1.0], dtype=torch.float32, device=omega.device)[:, None]
    q1 = _per_trajectory(plan.adjoint, w, omega, None, None).contiguous()
    q2 = _per_trajectory(plan.adjoint, w, (omega * flip).contiguous(), None, None).contiguous()
    N0, N1 = im_size
    kernel = torch.empty((nk, 2 * N0, 2 * N1), dtype=torch.complex64, device=omega.device)
    with torch.cuda.device(omega.device):
        ws = torch.empty(nk * 4 * N0 * N1 * 8, dtype=torch.uint8, device=omega.device)
        check(lib().pdu_toep_kernel_c64(h, q1.data_ptr(), q2.data_ptr(), kernel.data_ptr(), nk, scale, ws.data_ptr(),
                                        ws.numel(), stream_ptr()), "pdu_toep_kernel_c64")
    return kernel if omega.dim() == 3 else kernel[0]


# ----------------------------------------------------------------------------- conjugate gradient on the normal operator
def _cg_lam(lam, B: int, device: torch.device):
    """(device float32 lam or None for 0, lam_count).  A Python number becomes a one-entry tensor by a fill kernel."""
    if isinstance(lam, torch.Tensor):
        if not lam.is_cuda:
            raise PduError(f"lam is on {lam.device}: the pd_unet_b200 operators run on CUDA only (no CPU fallback)")
        if lam.dtype != torch.float32:
            raise TypeError(f"a tensor lam must be float32, got {lam.dtype}")
        if lam.numel() not in (1, B):
            raise ValueError(f"a tensor lam must have 1 or B = {B} entries, got {tuple(lam.shape)}")
        return lam.detach().reshape(-1).contiguous(), lam.numel()
    if isinstance(lam, bool) or not isinstance(lam, (int, float)):
        raise ValueError(f"lam must be a float >= 0 or a float32 CUDA tensor, got {type(lam).__name__}")
    if not float(lam) >= 0.0:
        raise ValueError(f"lam must be >= 0, got {lam}")
    if float(lam) == 0.0:
        return None, 1
    return torch.full((1,), float(lam), dtype=torch.float32, device=device), 1


def _toep_cg_solve(b, kernel, smaps, lam_dev, lam_count: int, x0, max_iter: int, tol: float, conj: bool) -> torch.Tensor:
    b, kernel, smaps, coils, sb = _toep_args(b, kernel, smaps, "b")
    B, _, N0, N1 = b.shape
    if x0 is not None:
        x0 = require_cuda(x0, torch.complex64, "x0")
        if x0.shape != b.shape:
            raise ValueError(f"x0 must have the shape of b {tuple(b.shape)}, got {tuple(x0.shape)}")
    x = torch.empty_like(b)
    if x.numel() == 0:
        return x
    with torch.cuda.device(b.device):
        tp = _toep_plan((N0, N1))
        h = tp.handle(b.device)
        L = lib()
        ws = torch.empty(int(L.pdu_toep_cg_workspace_bytes(h, B, coils, 1 if smaps is not None else 0)), dtype=torch.uint8,
                         device=b.device)
        check(L.pdu_toep_cg_c64(h, b.data_ptr(), x0.data_ptr() if x0 is not None else None, x.data_ptr(), kernel.data_ptr(),
                                kernel.shape[0], smaps.data_ptr() if smaps is not None else None, B, coils, sb,
                                lam_dev.data_ptr() if lam_dev is not None else None, lam_count, max_iter, tol, 1 if conj else 0,
                                ws.data_ptr(), ws.numel(), stream_ptr()), "pdu_toep_cg_c64")
    return x


class _ToepCgFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, b, lam_t, kernel, smaps, x0, lam_dev, lam_count, max_iter, tol):
        x = _toep_cg_solve(b, kernel, smaps, lam_dev, lam_count, x0, max_iter, tol, False)
        ctx.save_for_backward(kernel, x, smaps)
        ctx.cg = (lam_dev, lam_count, max_iter, tol)
        ctx.lam_shape = lam_t.shape if lam_t is not None else None
        return x

    @staticmethod
    def backward(ctx, g):
        kernel, x, smaps = ctx.saved_tensors
        lam_dev, lam_count, max_iter, tol = ctx.cg
        # implicit differentiation of x = M^-1 b, M = T + lam I: grad_b = M^-H g (the conj-kernel system), and
        # dx / dlam = -M^-1 x, so grad_lam = -Re <M^-H g, x> per lam entry
        gb = _toep_cg_solve(g.contiguous(), kernel, smaps, lam_dev, lam_count, None, max_iter, tol, True)
        glam = gs = None
        if ctx.needs_input_grad[1]:
            prod = (gb.conj() * x).real
            glam = -(prod.sum() if lam_count == 1 else prod.sum(dim=(1, 2, 3))).reshape(ctx.lam_shape)
        if smaps is not None and ctx.needs_input_grad[3]:
            # dx = -M^-1 (dM) x, so grad_S = -G(x, M^-H g) with G the ToepNufft map gradient
            gs = _toep_smaps_grad(x, gb, kernel, smaps, -1.0)
        return (gb if ctx.needs_input_grad[0] else None), glam, None, gs, None, None, None, None, None


def toep_cg(b: torch.Tensor, kernel: torch.Tensor, smaps: Optional[torch.Tensor] = None, lam=0.0,
            x0: Optional[torch.Tensor] = None, max_iter: int = 10, tol: float = 0.0) -> torch.Tensor:
    """Conjugate gradient on the Toeplitz normal operator: solves (T + lam I) x = b with T(v) = ToepNufft()(v, kernel,
    smaps=smaps), for every system of the batch at once, entirely on the device.

    b: complex64 [B, C, N0, N1], every (batch, channel) plane its own system; with smaps [1 or B, coils, N0, N1], b is
    [B, 1, N0, N1] and each batch element is one system (CG-SENSE).  kernel: [2 N0, 2 N1] or [1 or B, 2 N0, 2 N1] from
    calc_toeplitz_kernel.  lam: a float >= 0, or a float32 CUDA tensor with 1 or B entries (channels of a batch element
    share its lam; a tensor is not checked for sign, which would need a read-back).  x0: the warm start, shape of b;
    None starts from zero.  max_iter: iterations run, an int >= 0 (0 returns x0, or zeros).  tol >= 0: relative to
    ||b|| per system, like scipy's rtol.

    Per system, with float64 scalars and complex64 vectors:
        r = b - (T + lam) x0  (r = b without x0);  p = r;  rho = ||r||^2;  bb = ||b||^2
        repeat max_iter times:
            q = (T + lam) p;  pi = Re<p, q>
            if frozen or rho == 0 or pi <= 0:  freeze (x and r stay as they are from then on)
            alpha = rho / pi;  x += alpha p;  r -= alpha q;  rho' = ||r||^2
            if rho' <= tol^2 bb:  freeze
            p = r + (rho' / rho) p;  rho = rho'
    tol freezes a converged system but never ends the call early: every call runs max_iter iterations of device work,
    so a looser tol does not make it faster.  In exchange there is no host synchronisation and the whole solve can be
    captured in a CUDA graph.  The sums add in a fixed order without atomics, so a system's result is bit-identical
    whatever else is in the batch, however the batch is chunked, and under graph replay; no NaN or Inf is written (a
    zero right-hand side gives 0, a zero operator gives x0).

    Differentiable in b and in a tensor lam by implicit differentiation (the MoDL convention): grad_b solves the
    adjoint system (conj kernel) with the same lam, max_iter and tol, and grad_lam = -Re sum conj(grad_b) x per lam
    entry.  That is the gradient of the exact solution, which x approximates, not of the truncated iteration.  With
    smaps requiring a gradient, grad_S = -G(x, grad_b), G the ToepNufft map gradient (the adjoint system is solved even
    when b needs no gradient).  No gradient reaches kernel or x0."""
    if isinstance(max_iter, bool) or not isinstance(max_iter, int) or max_iter < 0:
        raise ValueError(f"max_iter must be an int >= 0, got {max_iter!r}")
    if isinstance(tol, bool) or not isinstance(tol, (int, float)) or not float(tol) >= 0.0:
        raise ValueError(f"tol must be a float >= 0, got {tol!r}")
    if not isinstance(b, torch.Tensor):
        raise TypeError("b must be a torch.Tensor")
    if not b.is_cuda:
        raise PduError(f"b is on {b.device}: the pd_unet_b200 operators run on CUDA only (no CPU fallback)")
    if b.dim() != 4:
        raise ValueError(f"b must be [B, C, N0, N1], got {tuple(b.shape)}")
    lam_dev, lam_count = _cg_lam(lam, b.shape[0], b.device)
    lam_t = lam if isinstance(lam, torch.Tensor) else None
    return _ToepCgFn.apply(b, lam_t, kernel, smaps, x0, lam_dev, lam_count, max_iter, float(tol))
