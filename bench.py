#!/usr/bin/env python
"""bench.py -- PD-UNet reconstruction throughput (slices/s) on BASELINE.json configs[1]:
parallel-beam CT, 256x256, 64 -> 512 views sinogram upsampling, batch 16 per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step is one inference pass of the unrolled PD-UNet over one batch of synthetic sparse-view
sinograms: per unrolled iteration one Radon forward projection (512 views), one dual CNN, one
ramp-filtered backprojection and one primal UNet, glued by the fused update kernels.  One JSON line
on rank 0.  `value`: inputs already in HBM, CUDA-event time summed over the K steps (L2 flushed
between steps outside the events), max over ranks.  `e2e`: the same pass from pinned host memory
to a host result.  `roofline`: the Radon forward-projection call timed live with CUDA events inside
those same K steps.  `cpu_baseline` / `--impl reference`: the CPU oracle port of the same model and the
same batch of 16 slices per step on all host cores -- `cpu_baseline` repeats the step until about 10 s are
on the clock, `--impl reference` runs at most one warm-up and K timed steps (the reference's own
operators, torch_radon, are CUDA-only and not mounted: SURVEY.md section 8c/8d).
`operators`: every hot-path operator alone (L2 flushed): Radon forward / adjoint / filter at configs[1], NUFFT
forward / adjoint at configs[0] and at the configs[3] per-GPU share, GSamples/s and fraction of the HBM roof.
`extras` (skip with --no-extras): the other BASELINE configs as model-level legs -- configs[0] radial-MRI inference
(256^2, 32 -> 256 spokes, one slice, CUDA graph), configs[2] fan-beam CT (512^2, 128 -> 1024 views, 8 slices per GPU),
configs[3] radial-MRI training step (320^2, 8 coils, 48 spokes; forward + loss + backward + Adam captured in one CUDA
graph, DDP's NCCL all-reduce inside it when --gpus N > 1).
`--dump-outputs DIR`: what the last timed step of each leg returned, as .npy files.  Inputs and weights are seeded, so
two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

N, A_SPARSE, UP, BATCH = 256, 64, 8, 16          # configs[1]
_STDOUT = None
A_FULL = A_SPARSE * UP
MODEL_KW = dict(n_iter=4, n_primal=4, n_dual=4, unet_base=32, unet_depth=3, dual_features=32)
METRIC = "PD-UNet recon slices/sec"
WORKLOAD = ("configs[1]: parallel-beam CT PD-UNet 256x256, 64->512 views sinogram upsampling, "
            "batch 16 per GPU (inference pass, 4 unrolled iterations)")


# ncu --set full numbers that bench.py does not measure itself (labelled as such in the JSON line)
STATIC_TRAFFIC = {"cold": 33912064 + 37888, "in_step": 52992 + 3401984,
                  "source": "profiles/r02_ncu_full_summary_fwd.md (cold: ncu flushes the caches, the kernel re-reads the two 16.9 MB "
                            "cell tensors) + profiles/r02_traffic_in_step.csv (--cache-control none: cells still in L2); ncu captures "
                            "of radon_fwd_quad_kernel<32,8,16,92,2,4,0>, dram read + write per launch; not re-measured by this run"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Polls SM clock and throttle reasons of one GPU while the timed region runs."""
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None

    def _poll(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self._nv is not None:
            self._thread = threading.Thread(target=self._poll, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def build_model(device):
    import pd_unet_b200 as pdu
    from pd_unet_b200.model import PrimalDualUNetCT
    angles = np.linspace(0.0, np.pi, A_FULL, endpoint=False)
    radon = pdu.Radon(N, angles)
    torch.manual_seed(1234)                      # random-init weights of the named architecture
    model = PrimalDualUNetCT(radon, upsample=UP, adjoint="fbp", **MODEL_KW).to(device).eval()
    return radon, model


def synthetic_sparse_sinograms(radon, device, batch, seed):
    """Sparse-view sinograms of Shepp-Logan-style phantoms, made with the operator itself."""
    from pd_unet_b200.phantoms import phantom_batch
    x = phantom_batch(batch, N, seed=seed).to(device)
    return radon.forward(x)[:, None, ::UP].contiguous()


def keep_output(dumps, name, t):
    """For --dump-outputs: a host float32 copy of what the last timed step returned (complex as trailing re/im pairs).
    Call it after the timed window has been synchronised: a captured graph's output is overwritten by its next replay."""
    if dumps is not None:
        t = t.detach()
        dumps[name] = (torch.view_as_real(t) if t.is_complex() else t).float().cpu()


def write_outputs(out_dir, dumps):
    os.makedirs(out_dir, exist_ok=True)
    for name, t in dumps.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


# ============================================================================= our arm
def run_ours(args):
    import pd_unet_b200 as pdu
    from pd_unet_b200 import parallel, radon as radon_mod
    from pd_unet_b200.graph import GraphedInference

    rank, world, local = parallel.init_distributed("nccl", graph_capture=not args.no_extras)
    if world != args.gpus:
        if rank == 0:
            print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; launch with torch.distributed.run",
                  file=sys.stderr)
        if world == 1 and args.gpus > 1:
            sys.exit(2)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    torch.backends.cudnn.benchmark = os.environ.get("PDU_BENCH_AUTOTUNE", "1") == "1"   # 0 for ncu launch lists
    radon, model = build_model(dev)
    sparse = synthetic_sparse_sinograms(radon, dev, BATCH, seed=100 + rank)      # resident in HBM
    host_in = sparse.cpu().pin_memory()
    host_out = torch.empty((BATCH, 1, N, N), dtype=torch.float32).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)                # > 126 MB L2

    def step(x):
        with torch.no_grad():
            return model(x)

    for _ in range(max(args.warmup, 3)):
        step(sparse)
    torch.cuda.synchronize()

    # ---- (1) eager pass: the forward projector timed live, with CUDA events, inside real steps
    op_events = []

    def hook(kind):
        if kind != "fwd":
            return None
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        op_events.append((s, e))
        return s, e

    ev0 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    pdu.launch_count(reset=True)
    radon_mod.EVENT_HOOK = hook
    for s, e in ev0:
        flush.zero_()
        s.record()
        step(sparse)
        e.record()
    torch.cuda.synchronize()
    radon_mod.EVENT_HOOK = None
    launches = pdu.launch_count()                      # our kernels in K steps (the graph replays the same launches)
    eager_ms = sum(s.elapsed_time(e) for s, e in ev0)
    fwd_ms = [s.elapsed_time(e) for s, e in op_events]

    # ---- (2) the timed region: the same step captured once as a CUDA graph and replayed
    use_graph = os.environ.get("PDU_BENCH_GRAPH", "1") == "1"
    graphed = GraphedInference(model, sparse, warmup=2) if use_graph else None

    def run_step():
        return graphed.replay() if use_graph else step(sparse)

    def e2e_step():
        if use_graph:
            y = graphed(host_in)                       # H2D into the captured input, replay
        else:
            y = step(host_in.to(dev, non_blocking=True))
        host_out.copy_(y, non_blocking=True)           # D2H of the reconstruction

    for _ in range(3):
        run_step()
    e2e_step()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    parallel.barrier()
    torch.cuda.synchronize()
    with ClockSampler(local) as clocks:
        for s, e in ev:
            flush.zero_()
            s.record()
            rec = run_step()
            e.record()
        torch.cuda.synchronize()
    dumps = {} if args.dump_outputs and rank == 0 else None
    keep_output(dumps, "reconstruction", rec)
    parallel.barrier()
    total_ms = parallel.max_over_ranks(sum(s.elapsed_time(e) for s, e in ev), dev)

    # ---- (3) end to end from pinned host memory to a host result
    ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    parallel.barrier()
    torch.cuda.synchronize()
    for s, e in ev2:
        flush.zero_()
        s.record()
        e2e_step()
        e.record()
    torch.cuda.synchronize()
    parallel.barrier()
    e2e_ms = parallel.max_over_ranks(sum(s.elapsed_time(e) for s, e in ev2), dev)

    # ---- operator microbenchmarks (each call alone, L2 flushed): GSamples/s and HBM fraction
    from pd_unet_b200 import _lib
    fwd_kernel = _lib.last_kernel("radon_fwd")         # what the dispatcher chose for the steps above
    ops = operator_microbench(radon, dev, flush) if rank == 0 else {}
    # ---- the other BASELINE configs as model-level legs (every rank takes part: the training leg is DDP)
    del graphed
    torch.cuda.empty_cache()
    extras = {} if args.no_extras else extra_legs(dev, flush, rank, world, local, args, dumps)

    if rank != 0:
        return
    if dumps is not None:
        write_outputs(args.dump_outputs, dumps)
    peak, peak_src = peaks()
    slices = BATCH * world * args.steps
    alg_bytes = 4.0 * BATCH * (N * N + A_FULL * N)               # DESIGN.md: 4 B (N^2 + A D) per call
    fwd_avg_ms = sum(fwd_ms) / len(fwd_ms)
    achieved = alg_bytes / (fwd_avg_ms * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": slices / (total_ms * 1e-3), "unit": "slices/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "dtype_note": "operators float32 throughout; cuDNN convolutions with TF32 allowed (PyTorch default, as the reference runs)",
        "config": {"workload": WORKLOAD, "image": N, "views_sparse": A_SPARSE, "views_full": A_FULL,
                   "batch_per_gpu": BATCH, "model": MODEL_KW, "weights": "random init (seed 1234)",
                   "parallelism": f"slice-sharded x{world}, no collective",
                   "launch": "CUDA graph replay of the whole step" if use_graph else "eager",
                   "ms_per_step_eager": eager_ms / args.steps,
                   "l2": "256 MiB write between steps, outside the events; activations (134 MB / feature map) exceed L2"},
        "e2e": {"value": slices / (e2e_ms * 1e-3), "unit": "slices/s", "h2d_bytes_per_step": host_in.numel() * 4,
                "d2h_bytes_per_step": host_out.numel() * 4},
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
        "roofline": {"bound": "hbm", "kernel": "pdu_radon_fwd_f32: " + fwd_kernel,       # pdu_last_kernel(): the dispatcher's choice in this run
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     # NOT measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of the projector kernel from
                     # a committed ncu --set full capture (see traffic_source).  ncu flushes the caches before every
                     # kernel, so it is the cold figure: the two 16.9 MB cell tensors quad_build_kernel has just written;
                     # inside a step they are still in L2 (traffic_in_step, --cache-control none).
                     "traffic": STATIC_TRAFFIC["cold"], "traffic_in_step": STATIC_TRAFFIC["in_step"],
                     "traffic_source": STATIC_TRAFFIC["source"],
                     "peak_source": peak_src, "algorithmic_bytes": alg_bytes, "avg_launch_ms": fwd_avg_ms,
                     "launches_timed": len(fwd_ms),
                     "gsamples_per_s": BATCH * A_FULL * N * N / (fwd_avg_ms * 1e-3) / 1e9,
                     "smem_roof_frac": (BATCH * A_FULL * N * N / (fwd_avg_ms * 1e-3)) / (148 * 8 * 1.965e9),
                     "note": "bound on-chip, not by HBM (43 samples per algorithmic byte): smem_roof_frac is samples/s "
                             "against the shared-memory roof of 8 bilinear samples/clk/SM (16 B/sample at 128 B/clk); "
                             "ncu (r02): L1/shared pipe 73 % busy (16 % of the wavefronts are bank conflicts of the 16-byte "
                             "cell loads), issue slots 71 % busy. DESIGN.md section 3"},
        "operators": ops,
        "extras": extras,
    }
    if not args.no_cpu and world == 1:                 # the CPU leg is reported at N = 1 only
        line["cpu_baseline"] = cpu_baseline()
    _STDOUT.restore()
    print(json.dumps(line), flush=True)


def operator_microbench(radon, dev, flush, reps=10):
    import pd_unet_b200 as pdu
    peak, _ = peaks()
    x = torch.rand(BATCH, N, N, device=dev)
    s = torch.rand(BATCH, A_FULL, N, device=dev)
    h = torch.rand(BATCH, 4, A_FULL, N, device=dev)

    def timed(fn):
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
            ts.append(a.elapsed_time(b))
        return statistics.median(ts)

    rb = 4.0 * BATCH * (N * N + A_FULL * N)
    out = {}
    from pd_unet_b200 import _lib
    from pd_unet_b200.data import radial_trajectory
    from pd_unet_b200.phantoms import coil_maps
    cases = [("radon_fwd", lambda: radon._project(x), rb, BATCH * A_FULL * N * N, "radon_fwd"),
             ("radon_adj", lambda: radon._backproject(s), rb, BATCH * N * N * A_FULL, "radon_adj"),
             ("filter", lambda: radon._filter(s, "ramp"), 4.0 * (2 * BATCH * A_FULL * N + N * N), None, "filter"),
             ("residual_slice", lambda: pdu.updates.residual_slice(h, h, 0), 4.0 * h.numel() * 3 + 4.0 * h.numel() / 4,
              None, None)]
    # NUFFT: configs[0] (256^2, one coil, one slice; the 32 measured spokes and the 256 of the upsampled grid) and the
    # configs[3] per-GPU share (320^2, 8 coils, batch 8, 48 spokes).  Algorithmic bytes 8 B C (N^2 + M) + 8 M (+ 8 C N^2 maps).
    keep = []
    for tag, n, coils, B, spokes in (("cfg1_32sp", 256, 1, 1, 32), ("cfg1_256sp", 256, 1, 1, 256), ("cfg4_share", 320, 8, 8, 48)):
        om = radial_trajectory(spokes, 2 * n, device=dev)
        M = om.shape[1]
        fw, ad = pdu.KbNufft((n, n)), pdu.KbNufftAdjoint((n, n))
        sm = coil_maps(coils, n)[None].to(dev) if coils > 1 else None
        img = torch.randn(B, 1, n, n, dtype=torch.complex64, device=dev)
        kd = torch.randn(B, coils, M, dtype=torch.complex64, device=dev)
        nb = 8.0 * B * coils * (n * n + M) + 8.0 * M + (8.0 * coils * n * n if coils > 1 else 0.0)
        taps = B * coils * M * 36
        keep.append((om, sm, img, kd, fw, ad))
        cases.append((f"nufft_fwd_{tag}", (lambda fw=fw, img=img, om=om, sm=sm: fw(img, om, smaps=sm, norm="ortho")), nb, taps, "nufft_fwd"))
        cases.append((f"nufft_adj_{tag}", (lambda ad=ad, kd=kd, om=om, sm=sm: ad(kd, om, smaps=sm, norm="ortho")), nb, taps, "nufft_adj"))
    for name, fn, nbytes, samples, op in cases:
        ms = timed(fn)
        out[name] = {"ms": ms, "GB/s": nbytes / ms / 1e6, "hbm_frac": nbytes / ms / 1e6 / peak, "algorithmic_bytes": nbytes}
        if samples:
            out[name]["GSamples/s"] = samples / ms / 1e6
        if op:
            out[name]["kernel"] = _lib.last_kernel(op)
    return out


# ============================================================================= the other BASELINE configs
def _timed_steps(run, flush, steps, dev):
    from pd_unet_b200 import parallel
    for _ in range(3):
        run()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    parallel.barrier()
    torch.cuda.synchronize()
    for a, b in ev:
        flush.zero_()
        a.record()
        run()
        b.record()
    torch.cuda.synchronize()
    parallel.barrier()
    return parallel.max_over_ranks(sum(a.elapsed_time(b) for a, b in ev), dev) / steps


def extra_legs(dev, flush, rank, world, local, args, dumps=None):
    """configs[0], configs[2] and configs[3] at model level (see the module docstring).  Every leg is weak scaling
    (fixed work per GPU); values are whole-job aggregates over the `world` GPUs, CUDA-event time, max over ranks.
    Each leg times --steps steps; with `dumps` (a dict) it also keeps what the last of them returned."""
    import pd_unet_b200 as pdu
    from pd_unet_b200 import data, parallel
    from pd_unet_b200.graph import GraphedInference, GraphedTrainingStep
    from pd_unet_b200.model import PrimalDualUNetCT, PrimalDualUNetMRI
    steps = args.steps
    out = {}
    # ---- configs[0]: radial-MRI inference, 256^2, 32 measured spokes regridded to 256, one slice per GPU
    n, sp_s, sp_f = 256, 32, 256
    torch.manual_seed(1234)
    mri = PrimalDualUNetMRI((n, n), sp_f, 2 * n, coils=1, **MODEL_KW).to(dev).eval()
    d = data.make_mri_batch((n, n), sp_s, 1, 1, seed=200 + rank, device=dev)
    om_full = data.radial_trajectory(sp_f, 2 * n, device=dev)
    dcf_full = pdu.calc_density_compensation_function(om_full, (n, n))
    fn = lambda kd: mri(kd, om_full, None, dcf_full, omega_sparse=d["omega"], dcf_sparse=d["dcf"])
    with torch.no_grad():
        g = GraphedInference(fn, d["kdata"], warmup=2)
    ms = _timed_steps(g.replay, flush, steps, dev)
    keep_output(dumps, "cfg1_mri_inference", g.static_out)
    out["cfg1_mri_inference"] = {"workload": "configs[0]: radial-MRI PD-UNet 256x256, 32 spokes regridded to 256 on the GPU (own NUFFT), "
                                             "1 slice per GPU, CUDA graph", "ms_per_step": ms, "slices_per_s": world / (ms * 1e-3)}
    del g, mri, d
    torch.cuda.empty_cache()
    # ---- configs[2]: fan-beam CT, 512^2, 128 -> 1024 views, 8 slices per GPU (batch 64 over 8 GPUs)
    n, a_s, up, b = 512, 128, 8, 8
    fan = pdu.RadonFanbeam(n, np.linspace(0.0, 2.0 * np.pi, a_s * up, endpoint=False), 2.0 * n)
    torch.manual_seed(1234)
    ct = PrimalDualUNetCT(fan, upsample=up, adjoint="fbp", **MODEL_KW).to(dev).eval()
    sparse = data.make_ct_batch(fan, b, up, seed=300 + rank, device=dev)["sino_sparse"]
    with torch.no_grad():
        g = GraphedInference(ct, sparse, warmup=2)
    ms = _timed_steps(g.replay, flush, steps, dev)
    keep_output(dumps, "cfg3_fan_ct_inference", g.static_out)
    out["cfg3_fan_ct_inference"] = {"workload": "configs[2]: fan-beam CT PD-UNet 512x512, 128->1024 views, 8 slices per GPU, CUDA graph",
                                    "ms_per_step": ms, "slices_per_s": b * world / (ms * 1e-3),
                                    "peak_mem_GiB": torch.cuda.max_memory_allocated(dev) / 2 ** 30}
    del g, ct, sparse, fan
    torch.cuda.empty_cache()
    # ---- configs[3]: radial-MRI training step, 320^2, 8 coils, 48 spokes, 2 slices per GPU, DDP when world > 1
    n, coils, sp, b = 320, 8, 48, 2
    torch.manual_seed(1234)
    m = PrimalDualUNetMRI((n, n), sp, 2 * n, coils=coils, n_iter=4, n_primal=4, n_dual=2 * coils, unet_base=32, unet_depth=3,
                          dual_features=32).to(dev)
    d = data.make_mri_batch((n, n), sp, coils, b, seed=400 + rank, device=dev)
    ddp = parallel.wrap_ddp(m, local, graph_capture=True)
    opt = torch.optim.Adam(ddp.parameters(), 1e-4, capturable=True)
    loss_fn = lambda o, t: (o - t).abs().pow(2).mean()
    step = GraphedTrainingStep(ddp, opt, loss_fn, (d["kdata"], d["omega"], d["smaps"], d["dcf"]), d["image"], warmup=3)
    ms = _timed_steps(step.graph.replay, flush, steps, dev)
    keep_output(dumps, "cfg4_mri_training_loss", step.static_loss)
    out["cfg4_mri_training"] = {"workload": "configs[3]: radial-MRI PD-UNet 320x320, 8 coils, 48 spokes, training step (forward + MSE + "
                                            "backward + Adam), 2 slices per GPU, one CUDA graph" + (", DDP NCCL all-reduce inside" if world > 1 else ""),
                                "ms_per_step": ms, "slices_per_s": b * world / (ms * 1e-3), "loss": float(step.static_loss.detach()),
                                "peak_mem_GiB": torch.cuda.max_memory_allocated(dev) / 2 ** 30}
    del step, ddp, opt, m, d
    torch.cuda.empty_cache()
    return out


# ============================================================================= CPU oracle port
def cpu_model_step(model64, sparse, trig, g):
    """The same unrolled pass on the host: torch CPU convolutions + the oracle's operators."""
    from oracle import c_port as oc          # OpenMP C restatement of oracle/radon.py (all host cores)
    from oracle import updates as ou
    m = model64
    gg = (ou.angular_upsample(sparse[:, 0], UP, "flip")[:, None] / m.op_scale).float()
    B = gg.shape[0]
    h = gg.new_zeros((B, m.n_dual, A_FULL, N))
    f = gg.new_zeros((B, m.n_primal, N, N))
    inv = 1.0 / m.op_scale
    with torch.no_grad():
        for i in range(m.n_iter):
            # K 0 = 0: like the CUDA arm, the first (zero) projection is not computed
            kf = oc.radon_forward(f[:, 0], trig, g)[:, None].to(gg.dtype) * inv if i > 0 else torch.zeros_like(gg)
            h = h + m.dual[i](torch.cat([h, kf, gg], 1))
            kth = oc.fbp(h[:, 0], trig, g)[:, None].to(gg.dtype) * inv
            f = f + m.primal[i](torch.cat([f, kth], 1))
    return f[:, :1]


def cpu_setup(sample_slices):
    import oracle
    from pd_unet_b200.model import PrimalDualUNet
    from pd_unet_b200.phantoms import phantom_batch
    angles = np.linspace(0.0, np.pi, A_FULL, endpoint=False)
    g = oracle.RadonGeom(n=N, n_angles=A_FULL, det_count=N)
    trig = oracle.trig_table(-angles)
    torch.manual_seed(1234)
    model = PrimalDualUNet(None, None, 1, 1, op_scale=float(N), **MODEL_KW).eval()      # same architecture, fp32 CPU
    gs = oracle.RadonGeom(n=N, n_angles=A_SPARSE, det_count=N)
    from oracle import c_port as oc
    sparse = oc.radon_forward(phantom_batch(sample_slices, N, seed=100), trig[::UP], gs).float()[:, None]
    return model, sparse, trig, g


CPU_NOTE = ("own CPU restatement (oracle/radon_c.c, OpenMP float64 operators + torch CPU fp32 convolutions), "
            "not the reference: torch_radon has no CPU path and is not mounted")


def use_all_host_cores():
    """torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU legs are meant to use the whole host."""
    from oracle import c_port as oc
    n = os.cpu_count() or 1
    torch.set_num_threads(n)
    oc.set_threads(n)


def cpu_cores():
    from oracle import c_port as oc
    return max(torch.get_num_threads(), oc.n_threads())


def cpu_baseline(sample_slices=BATCH, min_seconds=10.0, max_passes=6):
    """The whole batch-16 step on the host, repeated until about 10 s of CPU work are on the clock."""
    use_all_host_cores()
    model, sparse, trig, g = cpu_setup(sample_slices)
    cpu_model_step(model, sparse[:1], trig, g)           # warm the thread pools / page in
    t0 = time.perf_counter()
    passes = 0
    while passes < max_passes:
        cpu_model_step(model, sparse, trig, g)
        passes += 1
        if time.perf_counter() - t0 >= min_seconds:
            break
    dt = time.perf_counter() - t0
    return {"value": sample_slices * passes / dt, "unit": "slices/s", "cores": cpu_cores(), "kind": "port",
            "host_cpus": os.cpu_count(), "seconds": dt,
            "sample": f"{passes} pass(es) over the batch of {sample_slices} slices, full model (4 iterations, 512 views); " + CPU_NOTE}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = BATCH                               # the same batch of 16 slices per step as our arm
    use_all_host_cores()
    model, sparse, trig, g = cpu_setup(sample)
    warm = min(args.warmup, 1)                   # each step is seconds of CPU work
    for _ in range(warm):
        cpu_model_step(model, sparse, trig, g)
    done = args.steps
    t0 = time.perf_counter()
    for _ in range(done):
        rec = cpu_model_step(model, sparse, trig, g)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"reconstruction": rec.float()})
    v = sample * done / dt
    base = {"value": v, "unit": "slices/s", "cores": cpu_cores(), "kind": "port", "host_cpus": os.cpu_count(),
            "sample": f"{sample} slices per step, {done} step(s) timed; " + CPU_NOTE}
    _STDOUT.restore()
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "slices/s", "n_gpus": args.gpus, "steps": done,
        "warmup": warm, "ms_per_step": dt / done * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64 operators / f32 convolutions", "data": "synthetic",
        "config": {"workload": WORKLOAD, "image": N, "views_sparse": A_SPARSE, "views_full": A_FULL,
                   "batch_per_step": sample, "model": MODEL_KW},
        "cpu_baseline": base,
        "e2e": {"value": v, "unit": "slices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), flush=True)


class StdoutToStderr:
    """Route file descriptor 1 to stderr while the benchmark runs, so that libraries that print to stdout
    (NCCL's version banner, cuDNN warnings) cannot get in front of the ONE JSON line; restore() before printing."""

    def __init__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)

    def restore(self):
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        os.close(self._saved)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of every leg")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[0] / [2] / [3] model-level legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of each leg returned, on rank 0, as DIR/<name>.npy in float32 "
                         "(about 13 MB): reconstruction and, unless --no-extras, cfg1_mri_inference (re/im in the last "
                         "axis), cfg3_fan_ct_inference, cfg4_mri_training_loss; --impl reference writes its reconstruction")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    global _STDOUT
    _STDOUT = StdoutToStderr()
    if args.impl == "reference":
        run_reference(args)
    else:
        if int(os.environ.get("RANK", "0")) != 0:
            args.no_cpu = True
        run_ours(args)
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
