"""Coil-map gradients at the configs[3] share (8 batch elements x 8 coils x 320^2, 48 spokes x 640, DCF), smaps batch
1 and 8: the backward of KbNufft, KbNufftAdjoint, ToepNufft and toep_cg with and without the map gradient, the same
gradient through the ATen composition (the no-smaps operators around an ATen multiply / coil sum), and the forward
operators the map terms are compared with.  CUDA events, 256 MB buffer zeroed between timed calls (L2 flushed), median
of REPS; the card's name and power limit are read in the same run.
    python tools/prof_smaps_grad.py [REPS=21]   (prints the report; profiles/r05_smaps_grad_timings.txt is one)"""
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import pd_unet_b200 as pdu
from pd_unet_b200.phantoms import coil_maps

dev = "cuda:0"
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 21
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
B, COILS, N, SPOKES, READOUT = 8, 8, 320, 48, 640


def traj(spokes, readout):
    phi = np.arange(spokes) * (111.246117975 * np.pi / 180.0)
    r = (np.arange(readout) - readout / 2) * (2 * np.pi / readout)
    return torch.from_numpy(np.stack([(r[None] * np.sin(phi)[:, None]).reshape(-1),
                                      (r[None] * np.cos(phi)[:, None]).reshape(-1)]).astype(np.float32)).to(dev)


def timed(fn):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    return statistics.median(ts)


def crand(*shape):
    return torch.complex(torch.randn(*shape, device=dev), torch.randn(*shape, device=dev))


def backward_time(fn, inp, S, G, with_maps):
    """median us of autograd.grad of fn(inp, S) for inp (and S when with_maps), the forward done once outside"""
    i = inp.clone().requires_grad_(True)
    s = S.clone().requires_grad_(with_maps)
    out = fn(i, s)
    wrt = (i, s) if with_maps else (i,)
    return timed(lambda: torch.autograd.grad(out, wrt, G, retain_graph=True))


def main():
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        smi = f"nvidia-smi unavailable ({e})"
    print(f"device: {torch.cuda.get_device_name(0)} | nvidia-smi name, power limit, max SM clock: {smi}")
    print(f"shape: {B} x {COILS} coils x {N}^2, {SPOKES} spokes x {READOUT}, norm='ortho', DCF; REPS={reps}, L2 flushed")
    torch.manual_seed(0)
    om = traj(SPOKES, READOUT)
    M = om.shape[1]
    im = (N, N)
    w = pdu.calc_density_compensation_function(om, im).real.reshape(-1).contiguous()
    k = pdu.calc_toeplitz_kernel(om, im, weights=w, norm="ortho")
    lam = 0.1 * float(k.abs().max())
    fwd, adj, toep = pdu.KbNufft(im).to(dev), pdu.KbNufftAdjoint(im).to(dev), pdu.ToepNufft()
    x, y = crand(B, 1, N, N), crand(B, COILS, M)
    gy, gx = crand(B, COILS, M), crand(B, 1, N, N)
    ops = {
        "KbNufft": (lambda i, s: fwd(i, om, smaps=s, norm="ortho"), x, gy,
                    lambda i, s: fwd(i * s, om, norm="ortho")),
        "KbNufftAdjoint": (lambda i, s: adj(i, om, smaps=s, norm="ortho", kweight=w), y, gx,
                           lambda i, s: (adj(i, om, norm="ortho", kweight=w) * s.conj()).sum(1, keepdim=True)),
        "ToepNufft": (lambda i, s: toep(i, k, smaps=s), x, gx,
                      lambda i, s: (toep(i * s, k) * s.conj()).sum(1, keepdim=True)),
        "toep_cg (10 iterations)": (lambda i, s: pdu.toep_cg(i, k, smaps=s, lam=lam, max_iter=10), x, gx, None),
    }
    for sb in (1, B):
        S = (coil_maps(COILS, N).to(dev)[None] * (1.0 + 0.05 * crand(sb, COILS, N, N))).contiguous()
        print(f"\n== smaps batch {sb}")
        with torch.no_grad():
            t_adj = timed(lambda: adj(y, om, smaps=S, norm="ortho", kweight=w))
            t_app = timed(lambda: toep(x, k, smaps=S))
        print(f"  reference: one coil-map adjoint (KbNufftAdjoint forward) {t_adj:8.1f} us; one ToepNufft apply {t_app:8.1f} us")
        for name, (fn, inp, G, aten) in ops.items():
            t0 = backward_time(fn, inp, S, G, False)
            t1 = backward_time(fn, inp, S, G, True)
            line = f"  {name:24s} backward: input only {t0:8.1f} us, + maps {t1:8.1f} us, map term {t1 - t0:8.1f} us"
            if name in ("KbNufft", "KbNufftAdjoint"):
                line += f" = {(t1 - t0) / t_adj:4.2f} x one coil-map adjoint"
            elif name == "ToepNufft":
                line += f" = {(t1 - t0) / t_app:4.2f} x one apply"
            if aten is not None:
                ta = backward_time(aten, inp, S, G, True)
                line += f"; ATen composition (input + maps) {ta:8.1f} us"
            print(line)


if __name__ == "__main__":
    main()
