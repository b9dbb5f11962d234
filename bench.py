#!/usr/bin/env python
"""bench.py -- rays/s of the render_rays hot path (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--precision MODE] [--impl reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[1] -- a 400x400 lego-shape frame, 160 000
synthetic camera rays, N_samples=64 + N_importance=64, 8x256 MLP, fp32-parity arithmetic,
seeded default-init weights.  One step = one complete render_rays of the frame.
N > 1 (torchrun, one rank per GPU): weak scaling -- the job is N frames, each rank renders its
contiguous 160 000-ray slab and the rendered pixels (16 B/ray) reach every rank -- stored by the
compositing kernel itself into all ranks' frame buffers (NVSwitch multicast / NVLink P2P, CUDA
symmetric memory; distributed.PeerPixels), or all-gathered over NCCL with SNB_BENCH_EXCHANGE=nccl.

value  : rays/s, inputs resident in HBM, CUDA-event timed per step (L2 flushed between steps,
         outside the event pairs), max over ranks.
e2e    : same metric through the public API with HOST (pinned) rays: H2D of the rays and D2H
         of [rgb_fine, depth_fine] inside the timed region.
roofline: the fine-pass field kernel (2/3 of all FLOPs) timed alone with CUDA events.
cpu_baseline: the CPU oracle port (the reference is Python/torch; it cannot travel to the GPU
         box) on the host cores, on a bounded sample of the same rays.
--impl reference: only the CPU arm, same JSON schema, "impl": "reference".
--dump-outputs DIR: what render_rays returned in the last timed step (rank 0) as DIR/<key>.npy; see dump_outputs.
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
sys.dont_write_bytecode = True      # the tree may be read-only: the bench leaves it as build() left it

import torch  # noqa: E402

FLOP_PER_POINT = 2 * 593408          # SURVEY.md 8d (full head)
N_SAMPLES, N_IMPORTANCE = 64, 64
POINTS_PER_RAY = N_SAMPLES + (N_SAMPLES + N_IMPORTANCE)
METRIC = "rays/sec (64c+64f samples, 8x256 MLP)"
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


# stdout carries exactly ONE line, the JSON record: everything else that libraries write to fd 1 (NCCL's
# version banner, for one) is sent to stderr for the lifetime of the process.
_JSON_FD = None


def capture_stdout():
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    os.write(_JSON_FD if _JSON_FD is not None else 1, data)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            d["_source"] = "measured"
            return d
        except Exception:
            pass
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback"
    return d


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock / throttle reasons with NVML while the timed region runs."""

    def __init__(self, index: int):
        self.index, self.samples, self._stop = index, [], threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.max_sm = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                self.samples.append((sm, reasons, util))
            except Exception:
                pass
            time.sleep(0.05)

    def start(self):
        if self.ok:
            self.t.start()

    def stop(self):
        self._stop.set()
        if self.ok:
            self.t.join(timeout=1)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_sm, "reasons": [], "samples": 0}
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
                 "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80)}
        loaded = [s for s in self.samples if s[2] >= 50] or self.samples
        seen = set()
        for _, r, _ in loaded:
            for k, bit in names.items():
                if r & bit:
                    seen.add(k)
        return {"sm_mhz": statistics.median(s[0] for s in loaded), "sm_max_mhz": self.max_sm,
                "reasons": sorted(seen), "samples": len(loaded)}


# ----------------------------------------------------------------------------- CPU arm
_best_threads = None


def pick_threads(rays_cpu):
    """torch CPU GEMMs of this size stop scaling (and regress) long before 128 threads: try a few
    thread counts on a 256-ray sample and keep the fastest -- 'all the threads it can use'."""
    global _best_threads
    if _best_threads is None:
        from oracle import render_oracle as orc
        pc, pf = orc.default_init_params(0), orc.default_init_params(1)
        ncpu = os.cpu_count() or 1
        best = None
        for nt in sorted({ncpu, max(1, ncpu // 2), min(ncpu, 32), min(ncpu, 16), min(ncpu, 8)}):
            torch.set_num_threads(nt)
            r = rays_cpu[:256].contiguous()
            with torch.no_grad():
                orc.render_rays(pc, pf, r[:64], N_samples=N_SAMPLES, N_importance=N_IMPORTANCE, noise_std=0.0,
                                white_back=True)
                t0 = time.perf_counter()
                orc.render_rays(pc, pf, r, N_samples=N_SAMPLES, N_importance=N_IMPORTANCE, noise_std=0.0,
                                white_back=True)
                dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, nt)
        _best_threads = best[1]
    return _best_threads


def cpu_oracle_rate(rays_cpu, n_sample, repeats=1, budget_s=25.0):
    """rays/s of the CPU oracle port (oracle/render_oracle.py) on the first n_sample rays."""
    from oracle import render_oracle as orc
    torch.set_num_threads(pick_threads(rays_cpu))
    pc, pf = orc.default_init_params(0), orc.default_init_params(1)
    r = rays_cpu[:n_sample].contiguous()
    best, t_total, done = None, 0.0, 0
    with torch.no_grad():
        orc.render_rays(pc, pf, r[:256], N_samples=N_SAMPLES, N_importance=N_IMPORTANCE, noise_std=0.0,
                        white_back=True)
        while done < repeats and (done == 0 or t_total < budget_s):
            t0 = time.perf_counter()
            orc.render_rays(pc, pf, r, N_samples=N_SAMPLES, N_importance=N_IMPORTANCE, noise_std=0.0,
                            white_back=True)
            dt = time.perf_counter() - t0
            t_total += dt
            done += 1
            best = dt if best is None else min(best, dt)
    return r.shape[0] / best, torch.get_num_threads(), best


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's algorithm on the host CPU (oracle port: the reference is
    a Python package with missing deps (kornia, pytorch_lightning) that cannot travel to the GPU box)."""
    if rank != 0:
        return
    from sinnerf_b200 import synthetic
    rays = synthetic.frame_rays("lego", seed=0)
    n_sample = 2048
    for _ in range(max(0, args.warmup)):
        cpu_oracle_rate(rays, 512)
    times = []
    for _ in range(args.steps):
        rate, cores, dt = cpu_oracle_rate(rays, n_sample)
        times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    value = n_sample / (ms / 1e3)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": workload_config(args.gpus, "cpu-oracle"),
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": cores, "kind": "port",
                         "sample": f"first {n_sample} rays of the 400x400 frame per step, torch CPU fp32, "
                                   f"{cores} threads"},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(n_gpus, precision):
    return {"workload": "configs[1]: 400x400 lego-shape frame, 160000 rays/GPU, N_samples=64 N_importance=64, "
                        "8x256 MLP (use_new_activation), perturb=0 noise_std=0 white_back, seeded default-init weights",
            "rays_per_step_per_gpu": 160000, "global_rays_per_step": 160000 * n_gpus, "precision": precision,
            "parallelism": f"ray-sharded x{n_gpus}, the pixels of every slab delivered to every rank" if n_gpus > 1 else "single GPU",
            "l2": "256 MiB buffer written between timed steps (outside the per-step CUDA-event pairs)"}


# ----------------------------------------------------------------------------- GPU arm
DUMP_SAMPLE_ROWS = 32768


def dump_outputs(out_dir, res):
    """Write a render_rays result as out_dir/<key>.npy (float32), so that two builds can be compared output for output.
    rgb_* / depth_* are written whole; of the per-sample opacity_* arrays (123 MB for the 160 000-ray frame) the rows of
    a fixed seeded sample of DUMP_SAMPLE_ROWS rays, in ray order, the same rows in every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    n = res["rgb_fine"].shape[0]
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE_ROWS].sort().values
    for k, v in res.items():
        v = v.detach()
        if k.startswith("opacity_"):
            v = v[rows.to(v.device)]
        np.save(os.path.join(out_dir, f"{k}.npy"), v.float().cpu().numpy())


# ----------------------------------------------------------------------------- other BASELINE configs (extras)
def _fresh_models(dev, NeRF, default_init_params):
    models = []
    for seed in (0, 1):
        m = NeRF(use_new_activation=True)
        m.load_state_dict(default_init_params(seed))
        models.append(m.to(dev))
    return models


def _max_over_ranks(ms, dev, world):
    import torch.distributed as dist
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _timed_steps(fn, iters, flush, sync_all, dev, world):
    """mean ms per call: each call has its own CUDA-event pair, L2 flushed between calls, max over ranks of the sum."""
    evs = []
    sync_all()
    for _ in range(iters):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        evs.append((e0, e1))
    sync_all()
    return _max_over_ranks(sum(a.elapsed_time(b) for a, b in evs), dev, world) / iters


def bench_configs_2(models, emb, dev, lib, flush, sync_all, peaks):
    """BASELINE configs[2]: 504x378 LLFF shape, the 63x84 stride-4 ray patch (5 292 rays), 64+64 samples, bf16 MLP
    operands (fp32 accumulate), one B200.  rays/s of a complete render_rays + the fine-pass field kernel alone."""
    from sinnerf_b200 import _lib, rendering, synthetic
    if lib.snb_packed_weights_bytes(_lib.PRECISIONS["bf16"]) == 0:
        return {"unavailable": "bf16 mode not built"}
    rays = synthetic.patch_rays("llff", 63, 84, 4, seed=0).to(dev)
    n = rays.shape[0]

    def step():
        with torch.no_grad():
            return rendering.render_rays(models, emb, rays, N_SAMPLES, False, 0, 0, N_IMPORTANCE, 32768, False, precision="bf16")
    for _ in range(3):
        step()
    ms = _timed_steps(step, 20, flush, sync_all, dev, 1)
    with torch.no_grad():
        inter = rendering.render_rays(models, emb, rays, N_SAMPLES, False, 0, 0, N_IMPORTANCE, 32768, False, precision="bf16",
                                      _return_intermediates=True)["_inter"]
    z_f, raw_f = inter["z_fine"], inter["raw_fine"]
    S_f = N_SAMPLES + N_IMPORTANCE
    pid = _lib.PRECISIONS["bf16"]
    img = models[1].packed_weights(pid)

    def field_only():
        _lib.check(lib.snb_field_forward(_lib.ptr(img), pid, _lib.ptr(rays), _lib.ptr(z_f), n, S_f, 0, _lib.ptr(raw_f),
                                         _lib.stream_ptr(dev)), "snb_field_forward")
    for _ in range(3):
        field_only()
    kms = _timed_steps(field_only, 20, flush, sync_all, dev, 1)
    tf = FLOP_PER_POINT * n * S_f / (kms / 1e3) / 1e12
    peak = peaks.get("bf16_tflops") or FALLBACK_PEAKS["bf16_tflops"]       # a ~0.3 ms kernel timed alone: the burst figure
    return {"workload": "configs[2]: 63x84 stride-4 patch of a 504x378 LLFF-shape frame, 5292 rays, 64+64, bf16 operands / fp32 accumulate",
            "rays": n, "ms": ms, "rays_per_s": n / (ms / 1e3), "dtype": "bf16",
            "field_kernel_fine": {"ms": kms, "tflops_algorithmic": tf, "frac_of_bf16_peak": tf / peak, "peak": peak,
                                  "peak_source": f"MEASURED_PEAKS.json ({peaks['_source']}) bf16_tflops (burst)"}}


def make_exchange(rows, rows_per_rank, world, dev):
    """How the ranks' pixel slabs reach every rank.  Default: the compositing kernel stores them itself into all ranks'
    frame buffers (CUDA symmetric memory: one NVSwitch multicast address, else NVLink P2P addresses) -- distributed.PeerPixels;
    SNB_BENCH_EXCHANGE=nccl (or symmetric memory unavailable): the asynchronous NCCL all-gather of round 2 (PixelGather)."""
    from sinnerf_b200.distributed import PeerPixels, PixelGather
    if world == 1:
        return "none", None
    if os.environ.get("SNB_BENCH_EXCHANGE", "p2p") != "nccl":
        try:
            pp = PeerPixels(rows, dev)
            return ("kernel stores to the NVSwitch multicast address" if pp.multicast else "kernel stores to each peer (NVLink P2P)"), pp
        except Exception as e:      # noqa: BLE001 -- e.g. no P2P between the devices of this box
            sys.stderr.write(f"PeerPixels unavailable ({type(e).__name__}: {e}); using the NCCL all-gather\n")
    return "NCCL all-gather (async, double-buffered)", PixelGather(rows_per_rank, dev)


def bench_configs_3_strong(models, emb, dev, rank, world, precision, flush, sync_all):
    """BASELINE configs[3]: ONE 640x512 DTU-shape frame (327 680 rays, 64+64) strong-scaled over the ranks: every rank
    renders its contiguous slab and the pixels are all-gathered (16 B/ray).  The driver forms the speed-up from
    the per-N values."""
    from sinnerf_b200 import rendering, synthetic
    from sinnerf_b200.distributed import PeerPixels, render_frame_p2p, render_rays_sharded
    rays = synthetic.frame_rays("dtu", seed=0).to(dev)
    n = rays.shape[0]
    how, ex = make_exchange(n, -(-n // world), world, dev)

    def render_fn(r, sc=None):
        with torch.no_grad():
            return rendering.render_rays(models, emb, r, N_SAMPLES, False, 0, 0, N_IMPORTANCE, 32768, True, precision=precision,
                                         pixel_scatter=sc)

    if isinstance(ex, PeerPixels):
        def step():
            return render_frame_p2p(render_fn, rays, ex)

        def sync3():
            ex.wait_all()
            sync_all()
    else:
        how = "NCCL all-gather (blocking)" if world > 1 else how

        def step():
            return render_rays_sharded(render_fn, rays)
        sync3 = sync_all
    for _ in range(2):
        step()
    iters = 5
    ms = _timed_steps(step, iters, flush, sync3, dev, world)
    return {"workload": "configs[3]: 640x512 DTU-shape frame, 327680 rays, 64+64, rays sharded over the ranks, [rgb, depth] "
                        "(16 B/ray) of every slab delivered to every rank", "exchange": how, "scaling": "strong", "n_gpus": world,
            "rays_total": n, "rays_per_rank": -(-n // world), "ms": ms, "rays_per_s": n / (ms / 1e3), "precision": precision,
            "iters": iters}


def bench_configs_4_train(dev, rank, local_rank, world, precision, flush, sync_all, NeRF, Embedding, default_init_params):
    """BASELINE configs[4] (NeRF part): one SinNeRF training step per rank -- the four ray sets of
    models/sinnerf.py:304-307 (4 x 4096 rays, 64+64, perturb = 1, noise_std = 1) as ONE render_rays_multi pass,
    SmoothL1-depth / MSE-rgb evaluated inside the compositing kernels (8f-3), backward on tensor cores, DDP gradient
    all-reduce over NCCL when world > 1, FusedAdam step + weight re-pack (8f-4).  The ViT / discriminator branches are
    reference Python outside the hot path; their gradient enters as dL/d(rgb) of the two patch ray sets (a fixed
    linear functional here)."""
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP
    from sinnerf_b200 import rendering, synthetic
    from sinnerf_b200.optim import FusedAdam
    n_rays, calls = 4096, 4
    models = _fresh_models(dev, NeRF, default_init_params)
    emb = [Embedding(3, 10), Embedding(3, 4)]
    batches = [synthetic.random_rays("lego", n_rays, seed=1000 * rank + 100 + i).to(dev) for i in range(calls)]
    g = torch.Generator().manual_seed(rank)
    trgb = torch.rand(n_rays, 3, generator=g).to(dev)
    tdep = (torch.rand(n_rays, generator=g) * 4 + 2).to(dev)
    ext = [(torch.randn(n_rays, 3, generator=g) / n_rays).to(dev) for _ in range(2)]
    specs = [rendering.RayLosses(trgb, tdep), None, None, rendering.RayLosses(None, tdep)]

    class Step(torch.nn.Module):
        """stand-in for the LightningModule (models/sinnerf.py): owns both NeRFs, forward = the step's loss"""

        def __init__(self, ms):
            super().__init__()
            self.nerf_coarse, self.nerf_fine = ms

        def forward(self, _step):        # DDP's pre-forward needs at least one positional input
            res = rendering.render_rays_multi([self.nerf_coarse, self.nerf_fine], emb, batches, N_SAMPLES, False, 1.0, 1.0,
                                              N_IMPORTANCE, 32768, True, precision=precision, batch_losses=specs)
            loss = res[0]["loss_rgb"] + 0.1 * res[0]["loss_depth"]
            for k, w in zip((1, 2), ext):
                loss = loss + (res[k]["rgb_fine"] * w).sum() + (res[k]["rgb_coarse"] * w).sum()
            return loss

    mod = Step(models)
    net = DDP(mod, device_ids=[local_rank]) if world > 1 else mod
    opt = FusedAdam(models, lr=5e-4, precision=precision)

    def step():
        opt.zero_grad(set_to_none=True)
        net(0).backward()
        opt.step()
    for _ in range(3):
        step()
    torch.cuda.reset_peak_memory_stats(dev)
    iters = 5
    ms = _timed_steps(step, iters, flush, sync_all, dev, world)
    peak_gib = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    flops = 3 * FLOP_PER_POINT * n_rays * calls * POINTS_PER_RAY
    del net, opt, mod, models
    return {"workload": f"configs[4] (NeRF part): {calls} x {n_rays} rays per rank, 64+64, perturb=1 noise_std=1, render_rays_multi "
                        "forward + backward, fused per-ray losses, "
                        + ("DDP gradient all-reduce (NCCL), " if world > 1 else "") + "FusedAdam step + weight re-pack",
            "n_gpus": world, "ms_per_step": ms, "rays_per_s": n_rays * calls * world / (ms / 1e3), "precision": precision,
            "tflops_algorithmic_per_gpu": flops / (ms / 1e3) / 1e12, "peak_mem_gib": peak_gib, "iters": iters,
            "parallelism": f"ddp{world}" if world > 1 else "single GPU"}


def torch_cuda_baseline(rays_dev, default_init_params, n_prefix=8192):
    """The competitor a SinNeRF user has today (reference eval.py:141-155 on a GPU): the reference algorithm as stock
    PyTorch ops on this B200 -- oracle/render_oracle.py (the restatement pinned to the reference) on CUDA tensors,
    fp32 and with allow_tf32.  Informational row; not on any product path."""
    from oracle import render_oracle as orc
    dev = rays_dev.device
    pc = {k: v.to(dev) for k, v in default_init_params(0).items()}
    pf = {k: v.to(dev) for k, v in default_init_params(1).items()}
    r = rays_dev[:n_prefix].contiguous()
    out = {}
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    try:
        for tag, tf32 in (("fp32", False), ("tf32", True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            with torch.no_grad():
                for _ in range(2):
                    orc.render_rays(pc, pf, r, N_samples=N_SAMPLES, N_importance=N_IMPORTANCE, noise_std=0.0, white_back=True)
                torch.cuda.synchronize()
                best = None
                for _ in range(3):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    orc.render_rays(pc, pf, r, N_samples=N_SAMPLES, N_importance=N_IMPORTANCE, noise_std=0.0, white_back=True)
                    e1.record()
                    torch.cuda.synchronize()
                    ms = e0.elapsed_time(e1)
                    best = ms if best is None else min(best, ms)
            out[tag] = {"ms": best, "rays_per_s": r.shape[0] / (best / 1e3)}
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    out["sample"] = f"first {r.shape[0]} rays of the same 400x400 frame, 64+64, stock PyTorch CUDA ops (cuBLAS sgemm + ATen elementwise)"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("SINNERF_B200_BENCH_PRECISION", "auto"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[2]/[3]/[4] and stock-PyTorch rows")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what render_rays returned in the last timed step to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    capture_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch.distributed as dist
    from sinnerf_b200 import _lib, synthetic
    from sinnerf_b200 import build as _build
    from sinnerf_b200.distributed import pack_pixels, PeerPixels
    from sinnerf_b200.nerf import NeRF, Embedding
    from sinnerf_b200 import rendering
    from sinnerf_b200.synthetic import default_init_params  # noqa: E402  (seeded default-init weights)

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if rank == 0:
        _build.build()
    if world > 1:
        dist.barrier()
    lib = _lib.load()
    precision = args.precision
    if precision == "auto":
        precision = "f16x3" if lib.snb_packed_weights_bytes(_lib.PRECISIONS["f16x3"]) > 0 else "fp32"
    prec_id = _lib.precision_id(precision)

    models = []
    for seed in (0, 1):
        m = NeRF(use_new_activation=True)
        m.load_state_dict(default_init_params(seed))
        models.append(m.to(dev))
    emb = [Embedding(3, 10), Embedding(3, 4)]
    rays_cpu = synthetic.frame_rays("lego", seed=rank)          # this rank's frame (weak scaling)
    n = rays_cpu.shape[0]
    rays_pinned = rays_cpu.pin_memory()
    rays_dev = rays_cpu.to(dev)
    pix_host = torch.empty(n, 4).pin_memory()
    # every rank's pixels reach every rank: stored by the compositing kernel itself (PeerPixels) or all-gathered (PixelGather);
    # either way frame k's exchange overlaps render k + 1 (no per-step barrier)
    exchange_how, gather = make_exchange(n * world, n, world, dev)
    p2p = isinstance(gather, PeerPixels)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    rendering.DRAW_UNUSED_NOISE = True     # keep the reference's randn draws (rendering.py:224)

    def step(r, keep=None):
        k = gather.begin() if p2p else 0
        with torch.no_grad():
            res = rendering.render_rays(models, emb, r, N_SAMPLES, False, 0, 0, N_IMPORTANCE, 32768, True,
                                        precision=precision, pixel_scatter=gather.scatter(k, rank * n) if p2p else None)
        if keep is not None:
            keep["res"] = res
        pix = pack_pixels(res)
        if p2p:
            gather.commit(k)
        elif world > 1:
            gather.submit(pix)
        return pix

    def sync_all():
        if gather is not None:
            gather.wait_all()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, k):
        """k steps, each bracketed by its own event pair; L2 flushed between steps."""
        evs = []
        sync_all()
        for _ in range(k):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        sync_all()
        total_ms = sum(a.elapsed_time(b) for a, b in evs)
        tt = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    for _ in range(max(3, args.warmup)):
        step(rays_dev)
    sync_all()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    # with --dump-outputs each timed step keeps its result (dropping the previous one); written after the timed steps
    last = {} if args.dump_outputs and rank == 0 else None
    total_ms = timed(lambda: step(rays_dev, last), args.steps)
    if last is not None:
        dump_outputs(args.dump_outputs, last.pop("res"))

    def e2e_step():
        r = rays_pinned.to(dev, non_blocking=True)
        pix = step(r)
        pix_host.copy_(pix, non_blocking=True)

    for _ in range(2):
        e2e_step()
    e2e_ms = timed(e2e_step, args.steps)
    # ---- dominant kernel alone: the fine-pass field kernel (128 samples/ray)
    S_f = N_SAMPLES + N_IMPORTANCE
    with torch.no_grad():
        inter = rendering.render_rays(models, emb, rays_dev, N_SAMPLES, False, 0, 0, N_IMPORTANCE, 32768, True,
                                      precision=precision, _return_intermediates=True)["_inter"]
    z_f, raw_f = inter["z_fine"], inter["raw_fine"]
    img_f = models[1].packed_weights(prec_id)

    def field_only():
        _lib.check(lib.snb_field_forward(_lib.ptr(img_f), prec_id, _lib.ptr(rays_dev), _lib.ptr(z_f), n, S_f, 0,
                                         _lib.ptr(raw_f), _lib.stream_ptr(dev)), "snb_field_forward")

    for _ in range(2):
        field_only()
    kern_ms = timed(field_only, max(3, min(args.steps, 10))) / max(3, min(args.steps, 10))
    clocks = sampler.stop() if sampler else None

    # ---- the other BASELINE configs, outside the headline timed region (extra keys of the same JSON line)
    extra = {}
    if not args.no_extras:
        peaks_x = load_peaks()
        if world == 1:
            extra["configs_2"] = bench_configs_2(models, emb, dev, lib, flush, sync_all, peaks_x)
        extra["configs_3_strong"] = bench_configs_3_strong(models, emb, dev, rank, world, precision, flush, sync_all)
        extra["configs_4_ddp"] = bench_configs_4_train(dev, rank, local_rank, world, precision, flush, sync_all, NeRF, Embedding,
                                                       default_init_params)
        if world == 1:
            extra["torch_cuda_baseline"] = torch_cuda_baseline(rays_dev, default_init_params)

    if rank == 0:
        peaks = load_peaks()
        ms_per_step = total_ms / args.steps
        value = n * world / (ms_per_step / 1e3)
        e2e_value = n * world / ((e2e_ms / args.steps) / 1e3)
        kern_tflops = FLOP_PER_POINT * n * S_f / (kern_ms / 1e3) / 1e12
        # the kernel is timed alone but in a back-to-back loop of tens of ms each: the power-capped
        # ("sustained") cuBLAS figure is the comparable denominator
        tensor_peak = peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops")
        # tensor-core modes fold the 256x256 bottleneck into the direction layer at pack time, so they
        # execute (593408 - 65536) MACs per point and product; the split modes issue 3 products
        passes = (3 if precision.endswith("x3") else 1) * (593408 - 65536) / 593408
        traffic = None
        tp = os.path.join(ROOT, "profiles", "field_traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get(precision)
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": {"fp32": "fp32 (FFMA)", "f16x3": "fp32-parity: fp16 hi/lo split x3 on tcgen05, fp32 accumulate",
                      "bf16x3": "bf16 hi/lo split x3 on tcgen05, fp32 accumulate",
                      "bf16": "bf16 operands, fp32 accumulate"}[precision],
            "data": "synthetic",
            "config": workload_config(world, precision),
            "exchange": exchange_how,
            "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": n * 32 * world,
                    "d2h_bytes_per_step": n * 16 * world, "ms_per_step": e2e_ms / args.steps},
            # per render_rays: sample_coarse, field, composite, importance_merge, field, composite + per model the
            # weight-image check kernel and the two (conditional, normally empty) pack kernels
            "gpu_launches": 12 * args.steps,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "fine-pass field kernel (160000 rays x 128 samples)",
                         "achieved": kern_tflops, "peak": tensor_peak, "unit": "TFLOP/s",
                         "frac": kern_tflops / tensor_peak if tensor_peak else None, "traffic": traffic,
                         "executed_tflops": kern_tflops * passes if precision != "fp32" else None,
                         "frac_executed": kern_tflops * passes / tensor_peak if (tensor_peak and precision != "fp32") else None,
                         "peak_source": f"MEASURED_PEAKS.json ({peaks['_source']}), dense bf16 cuBLAS, sustained",
                         "ms_per_launch": kern_ms,
                         "flops": "algorithmic 2*593408 per point (SURVEY 8d); "
                                  + ("executed MMA flops: 3 products (hi*hi + hi*lo + lo*hi) x 0.89 (bottleneck folded into the dir layer)" if precision.endswith("x3")
                                     else "FFMA pipe, not tensor cores" if precision == "fp32" else "single pass")},
        }
        line["roofline"]["traffic_source"] = ("static: dram__bytes_read+write of one ncu --set full capture of this kernel at this "
                                              "size (profiles/field_traffic.json), not re-measured in this run")
        if extra:
            line["extra"] = extra
        if not args.no_cpu_baseline and world == 1:
            rate, cores, dt = cpu_oracle_rate(rays_cpu, 2048)
            line["cpu_baseline"] = {"value": rate, "unit": "rays/s", "cores": cores, "kind": "port",
                                    "sample": f"first 2048 rays of the same frame, one pass ({dt:.1f} s), "
                                              f"oracle/render_oracle.py on torch CPU fp32"}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
