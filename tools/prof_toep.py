"""Toeplitz normal operator (ToepNufft) against the NUFFT pair KbNufftAdjoint(KbNufft(x), kweight=w) -- the library's
default paths -- on the configs[3] share and other shapes; per-launch device times of the apply from torch.profiler;
the one-time kernel build.  CUDA events, 256 MB buffer zeroed between timed calls (L2 flushed), median of REPS.
    python tools/prof_toep.py [REPS=21]"""
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import pd_unet_b200 as pdu
from pd_unet_b200 import _lib
from pd_unet_b200.phantoms import coil_maps

dev = "cuda:0"
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 21
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def traj(spokes, readout):
    phi = np.arange(spokes) * (111.246117975 * np.pi / 180.0)
    r = (np.arange(readout) - readout / 2) * (2 * np.pi / readout)
    return torch.from_numpy(np.stack([(r[None] * np.sin(phi)[:, None]).reshape(-1),
                                      (r[None] * np.cos(phi)[:, None]).reshape(-1)]).astype(np.float32)).to(dev)


def timed(fn, n=None):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n or reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    return statistics.median(ts), min(ts), max(ts)


def per_launch(fn):
    """device time per kernel name (mean over 5 calls) from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            flush.zero_()
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if any(s in ev.key for s in ("tz_", "ff_rows", "pfft_", "crop_apod")):
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
            out[ev.key] = t / max(1, ev.count)
    return out


try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as e:  # noqa: BLE001
    smi = f"nvidia-smi unavailable ({e})"
print(f"device: {torch.cuda.get_device_name(0)} | nvidia-smi name, power limit, max SM clock: {smi}")
print(f"method: CUDA events around one call, 256 MB buffer zeroed before each call (L2 flushed), median (min / max) of {reps}")
print()

# name, N, coils (0: no coil maps, one channel), batch, spokes
CASES = (("configs[3] share, 64 planes of 320^2 (8 x 8 coils), 48 spokes", 320, 8, 8, 48),
         ("configs[3] training share, 16 planes of 320^2 (2 x 8 coils), 48 spokes", 320, 8, 2, 48),
         ("configs[0], 1 plane of 256^2, 256 spokes", 256, 0, 1, 256),
         ("dense, 16 planes of 512^2, 1024 spokes", 512, 0, 16, 1024),
         ("2 planes of 1024^2, 512 spokes", 1024, 0, 2, 512))
for name, n, coils, B, spokes in CASES:
    im = (n, n)
    om = traj(spokes, 2 * n)
    w = pdu.calc_density_compensation_function(om, im, num_iterations=4)
    wr = w.real.reshape(-1).contiguous()
    sm = coil_maps(coils, n)[None].to(dev) if coils else None
    x = torch.randn(B, 1, n, n, dtype=torch.complex64, device=dev)
    A, AH, T = pdu.KbNufft(im), pdu.KbNufftAdjoint(im), pdu.ToepNufft()
    build = timed(lambda: pdu.calc_toeplitz_kernel(om, im, weights=w, norm="ortho"), 5)
    k = pdu.calc_toeplitz_kernel(om, im, weights=w, norm="ortho")
    y = A(x, om, smaps=sm, norm="ortho")
    t_f = timed(lambda: A(x, om, smaps=sm, norm="ortho"))
    t_a = timed(lambda: AH(y, om, smaps=sm, norm="ortho", kweight=wr))
    t_pair = timed(lambda: AH(A(x, om, smaps=sm, norm="ortho"), om, smaps=sm, norm="ortho", kweight=wr))
    t_toep = timed(lambda: T(x, k, smaps=sm, norm="ortho"))
    path = _lib.last_kernel("toep")
    ref = AH(A(x, om, smaps=sm, norm="ortho"), om, smaps=sm, norm="ortho", kweight=wr)
    got = T(x, k, smaps=sm, norm="ortho")
    err = float((got - ref).norm() / ref.norm())
    print(f"== {name}  (M = {om.shape[1]})")
    print(f"   KbNufft forward            {t_f[0]:9.1f} us  ({t_f[1]:.1f} / {t_f[2]:.1f})")
    print(f"   KbNufftAdjoint (kweight)   {t_a[0]:9.1f} us  ({t_a[1]:.1f} / {t_a[2]:.1f})")
    print(f"   pair, one timed window     {t_pair[0]:9.1f} us  ({t_pair[1]:.1f} / {t_pair[2]:.1f})")
    print(f"   ToepNufft apply            {t_toep[0]:9.1f} us  ({t_toep[1]:.1f} / {t_toep[2]:.1f})   "
          f"= {t_toep[0] / t_pair[0]:.2f} x the pair")
    print(f"   calc_toeplitz_kernel       {build[0]:9.1f} us  (one-time build, median of 5)")
    print(f"   rel-L2 Toeplitz vs pair    {err:.2e}")
    print(f"   path: {path}")
    for kname, t in per_launch(lambda: T(x, k, smaps=sm, norm="ortho")).items():
        print(f"     {t:9.1f} us  {kname[:110]}")
    print(flush=True)
