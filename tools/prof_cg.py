"""toep_cg (conjugate gradient on the Toeplitz normal operator) on the cases of tools/prof_toep.py: the ToepNufft apply,
microseconds per CG iteration taken as (t(30) - t(10)) / 20 so that set-up drops out, per-launch device times of the
CG kernels from torch.profiler, launches per iteration, and the same algorithm written with ToepNufft and ATen ops
(no .item()), eager and captured in a CUDA graph.  CUDA events, 256 MB buffer zeroed between timed calls (L2
flushed), median of REPS.
    python tools/prof_cg.py [REPS=21]"""
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
ITERS = (10, 30)


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
    return statistics.median(ts)


def per_launch(fn):
    """device time per kernel name (mean per launch over 3 calls) from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            flush.zero_()
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if any(s in ev.key for s in ("cg_", "tz_", "ff_rows", "pfft_", "crop_apod")):
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
            out[ev.key] = (t / max(1, ev.count), ev.count)
    return out


def aten_cg(b, k, sm, lam, iters, tol=0.0):
    """The algorithm of include/pdu.h with ToepNufft and ATen ops: float64 scalars per system, no host read-back."""
    T = pdu.ToepNufft()

    def dot(u, v):
        return (u.conj() * v).real.to(torch.float64).sum(dim=(-2, -1), keepdim=True)

    x = torch.zeros_like(b)
    r = b.clone()
    p = r.clone()
    rho = dot(r, r)
    bb = rho.clone()
    frozen = torch.zeros_like(rho, dtype=torch.bool)
    zero = torch.zeros_like(rho)
    for _ in range(iters):
        q = T(p, k, smaps=sm) + lam * p
        pi = dot(p, q)
        stop = frozen | (rho == 0) | (pi <= 0)
        alpha = torch.where(stop, zero, rho / pi).to(torch.float32)
        x = x + alpha * p
        r = r - alpha * q
        rho_new = dot(r, r)
        frozen = stop | (rho_new <= tol * tol * bb)
        beta = torch.where(frozen, zero, rho_new / rho).to(torch.float32)
        p = torch.where(frozen, p, r + beta * p)
        rho = torch.where(frozen, rho, rho_new)
    return x


def graphed(fn):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g.replay


try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as e:  # noqa: BLE001
    smi = f"nvidia-smi unavailable ({e})"
print(f"device: {torch.cuda.get_device_name(0)} | nvidia-smi name, power limit, max SM clock: {smi}")
print(f"method: CUDA events around one call, 256 MB buffer zeroed before each call (L2 flushed), median of {reps}; "
      f"per iteration = (t({ITERS[1]}) - t({ITERS[0]})) / {ITERS[1] - ITERS[0]}")
print()

# name, N, coils (0: no coil maps, one channel), batch, spokes -- the cases of tools/prof_toep.py
CASES = (("configs[3] share, 8 systems of 8 coils x 320^2 (64 planes), 48 spokes", 320, 8, 8, 48),
         ("configs[3] training share, 2 systems of 8 coils x 320^2 (16 planes), 48 spokes", 320, 8, 2, 48),
         ("configs[0], 1 system of 256^2, 256 spokes", 256, 0, 1, 256),
         ("dense, 16 systems of 512^2, 1024 spokes", 512, 0, 16, 1024),
         ("2 systems of 1024^2, 512 spokes", 1024, 0, 2, 512))
for name, n, coils, B, spokes in CASES:
    im = (n, n)
    om = traj(spokes, 2 * n)
    w = pdu.calc_density_compensation_function(om, im, num_iterations=4)
    sm = coil_maps(coils, n)[None].to(dev) if coils else None
    k = pdu.calc_toeplitz_kernel(om, im, weights=w, norm="ortho")
    b = torch.randn(B, 1, n, n, dtype=torch.complex64, device=dev)
    T = pdu.ToepNufft()
    lam = 0.05 * float(k.abs().max())
    t_apply = timed(lambda: T(b, k, smaps=sm, norm="ortho"))
    t_cg = {m: timed(lambda m=m: pdu.toep_cg(b, k, smaps=sm, lam=lam, max_iter=m)) for m in ITERS}
    path = _lib.last_kernel("cg")
    launches = {}
    for m in ITERS:
        pdu.launch_count(reset=True)
        pdu.toep_cg(b, k, smaps=sm, lam=lam, max_iter=m)
        launches[m] = pdu.launch_count()
    t_aten = {m: timed(lambda m=m: aten_cg(b, k, sm, lam, m)) for m in ITERS}
    t_graph = {m: timed(graphed(lambda m=m: aten_cg(b, k, sm, lam, m))) for m in ITERS}
    x_own = pdu.toep_cg(b, k, smaps=sm, lam=lam, max_iter=ITERS[1])
    x_aten = aten_cg(b, k, sm, lam, ITERS[1])
    diff = float((x_own - x_aten).norm() / x_aten.norm())
    d = ITERS[1] - ITERS[0]

    def it(t):
        return (t[ITERS[1]] - t[ITERS[0]]) / d

    print(f"== {name}  (M = {om.shape[1]}, lam = 0.05 max|kernel|)")
    print(f"   ToepNufft apply                 {t_apply:9.1f} us")
    print(f"   toep_cg  {ITERS[0]} / {ITERS[1]} iterations      {t_cg[ITERS[0]]:9.1f} / {t_cg[ITERS[1]]:.1f} us")
    print(f"   toep_cg per iteration           {it(t_cg):9.1f} us  = {it(t_cg) / t_apply:.2f} x the apply")
    print(f"   ATen CG per iteration, eager    {it(t_aten):9.1f} us")
    print(f"   ATen CG per iteration, graph    {it(t_graph):9.1f} us")
    print(f"   launches per iteration          {(launches[ITERS[1]] - launches[ITERS[0]]) / d:9.1f}  "
          f"(set-up {launches[ITERS[0]] - ITERS[0] * (launches[ITERS[1]] - launches[ITERS[0]]) // d})")
    print(f"   rel-L2 toep_cg vs ATen CG, {ITERS[1]} it  {diff:.2e}")
    print(f"   path: {path}")
    for kname, (t, cnt) in per_launch(lambda: pdu.toep_cg(b, k, smaps=sm, lam=lam, max_iter=ITERS[0])).items():
        print(f"     {t:9.1f} us x {cnt // 3:3d}  {kname[:100]}")
    print(flush=True)
