#!/usr/bin/env python
"""bench.py — ControlLoRA training throughput on B200 (the BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this framework (one process per GPU; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm's CPU path (oracle port) on host cores
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR    # + what the last timed step computed, as DIR/*.npy

One "step" = hint-encoder fwd + SD-1.5 UNet fwd + MSE + backward (dX, LoRA dA/dB, hint-encoder dW) + gradient
all-reduce (N > 1) + clip_grad_norm + AdamW, on synthetic 512x512 inputs (64x64 latents, 77x768 text states), batch 8
per GPU, random-init weights of the SD-1.5 / ControlLoRA architecture (no checkpoints are reachable offline).
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True      # the benchmark leaves the tree it runs from as it found it (it may be read-only)

METRIC = "train_images_per_sec_512px_bs8_per_gpu"
UNIT = "images/s"
# algorithmic work per image (SURVEY.md §8d / BASELINE.md §2)
GFLOP_PER_IMAGE_STEP = 1794.0


def gemm_traffic_per_launch():
    """DRAM bytes per gemm_tc_kernel launch (dram__bytes_read.sum + dram__bytes_write.sum averaged over the GEMM launches of
    one training step) from the committed ncu capture profiles/r01_gemm_traffic.json; None when the file is missing."""
    try:
        root = Path(__file__).resolve().parent / "profiles"
        f = root / "r02_gemm_traffic.json"
        d = json.loads((f if f.exists() else root / "r01_gemm_traffic.json").read_text())
        return float(d["bytes_per_launch"])
    except Exception:
        return None


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="diffusiondb-canny-v2", help="ControlLoRA config name (controllora_b200.configs.NAMED)")
    ap.add_argument("--batch", type=int, default=8, help="per-GPU batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying the captured CUDA graph")
    ap.add_argument("--no-aux", action="store_true", help="skip the auxiliary numbers (denoise C3/C5, drop-in path, per-shape GEMM table)")
    ap.add_argument("--aux-only", default=None, choices=["train_from_pixels"],
                    help="run ONE auxiliary measurement in this process and print its JSON (bench.py runs it as an isolated child process)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one computed (loss, gradient norm, parameters and AdamW moments "
                         "after the update) as float32 DIR/<name>.npy; the inputs and initial weights are seeded, so two builds can be "
                         "compared output for output")
    return ap.parse_args()


def synth_inputs(torch, B, seed_off=0, device="cpu"):
    """SURVEY.md §8d synthetic tensors: latents / text states ~ N(0,1), canny-like {-1,+1} guide with ~8% edge pixels."""
    g = lambda s: torch.Generator().manual_seed(s + 1000 * seed_off)
    x = torch.randn(B, 4, 64, 64, generator=g(0))
    t = torch.randint(0, 1000, (B,), generator=g(1)).float()
    e = torch.randn(B, 77, 768, generator=g(2))
    edge = (torch.rand(B, 1, 512, 512, generator=g(3)) < 0.08).float() * 2 - 1
    guide = edge.expand(B, 3, 512, 512).contiguous()
    tgt = torch.randn(B, 4, 64, 64, generator=g(4))
    return x, t, e, guide, tgt


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe), polled from a thread."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0, period_s=0.02):
        self.idx, self.period = gpu_index, period_s
        self.lines, self.stop_flag, self.t = [], threading.Event(), None

    def _poll(self):
        cmd = ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.idx)]
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(cmd, capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.lines.append(out.splitlines()[0])
            except Exception:
                pass
            self.stop_flag.wait(self.period)

    def start(self):
        self.t = threading.Thread(target=self._poll, daemon=True)
        self.t.start()

    def stop(self):
        self.stop_flag.set()
        if self.t is not None:
            self.t.join(timeout=6)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower() == "active":
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi returned no samples"], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw), "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md: 1.4 PF sustained)"


# ------------------------------------------------------------------------------------------------------ CPU oracle arm
_CPU_THREADS = None


def pick_cpu_threads(torch) -> int:
    """Use the thread count that is actually fastest for this workload's kernels on the host: torch's CPU conv / matmul
    slow down badly when oversubscribed (128 threads measured 14x slower than 8 on the GPU box's host)."""
    global _CPU_THREADS
    if _CPU_THREADS is not None:
        return _CPU_THREADS
    ncpu = os.cpu_count() or 1
    x = torch.randn(1, 320, 64, 64)
    w = torch.randn(320, 320, 3, 3)
    a = torch.randn(4096, 320)
    b = torch.randn(320, 1280)
    best, best_t = 1, float("inf")
    for n in sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu}):
        torch.set_num_threads(n)
        for _ in range(2):
            torch.nn.functional.conv2d(x, w, padding=1); a @ b
        t0 = time.perf_counter()
        for _ in range(5):
            torch.nn.functional.conv2d(x, w, padding=1); a @ b
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = n, dt
    _CPU_THREADS = best
    return best


def cpu_train_step_factory(config_name: str):
    """The reference algorithm on the host cores: oracle port of diffusers' UNet + models.py (oracle/), fp32, one image."""
    import torch
    from oracle import models_ref as MR
    from oracle import unet_ref as UR
    from controllora_b200.configs import NAMED

    torch.set_num_threads(pick_cpu_threads(torch))
    unet = UR.UNet2DConditionModel()
    UR.init_synthetic_(unet, seed=1)
    unet.requires_grad_(False)
    cl = MR.ControlLoRA.from_config(NAMED[config_name])
    MR.randomize_lora_up_(cl, seed=3)
    MR.wire_processors(unet, cl)
    opt = torch.optim.AdamW(cl.parameters(), lr=1e-4, betas=(0.9, 0.999), weight_decay=1e-2, eps=1e-8)
    x, t, e, guide, tgt = synth_inputs(torch, 1)

    def step():
        cl(guide)
        loss = torch.nn.functional.mse_loss(unet(x, t.long(), e).sample, tgt)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(cl.parameters(), 1.0)
        opt.step()
        opt.zero_grad()
        return float(loss)

    return step


def cpu_baseline(config_name: str, budget_s: float = 25.0, max_steps: int = 2):
    step = cpu_train_step_factory(config_name)
    t0 = time.time()
    step()                      # warm-up (allocator, thread pool)
    warm = time.time() - t0
    n = 1 if warm > budget_s / 2 else max_steps
    t0 = time.time()
    for _ in range(n):
        step()
    dt = (time.time() - t0) / n
    import torch
    return {"value": 1.0 / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n} full train step(s) of ONE 512x512 image (batch 1) through the fp32 oracle port (oracle/), "
                      f"torch CPU with {torch.get_num_threads()} threads (fastest of a sweep up to {os.cpu_count()} logical CPUs); {dt:.1f} s/step"}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    step = cpu_train_step_factory(a.config)
    t0 = time.time()
    step()
    first = time.time() - t0
    budget = 150.0
    w_eff = 0 if first > 30 else min(a.warmup, 1)
    for _ in range(w_eff):
        step()
    k_eff = max(1, min(a.steps, int(budget / max(first, 1e-3))))
    t0 = time.time()
    for _ in range(k_eff):
        step()
    dt = (time.time() - t0) / k_eff
    v = 1.0 / dt
    out = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": k_eff, "warmup": w_eff + 1,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{a.config} ControlLoRA train step, SD-1.5 UNet 512x512 (64x64 latents), CPU sample = batch 1"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": _CPU_THREADS, "kind": "port",
                         "sample": f"{k_eff} timed train step(s) of one 512x512 image each ({a.steps} requested; bounded to ~150 s), "
                                   f"fp32 oracle port of the reference (diffusers is not installable offline), {_CPU_THREADS} threads "
                                   f"(fastest of a sweep up to {os.cpu_count()} logical CPUs)"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------------ auxiliary GPU numbers
def _randomize_up(torch, module, dev, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for n_, p_ in module.named_parameters():
            if n_.endswith("up.weight"):
                p_.copy_((0.02 * torch.randn(p_.shape, generator=g)).to(p_.device))


def aux_denoise(torch, cb, unet, which):
    """BASELINE.json configs 3 and 5 through controllora_b200.sampler.GraphedSampler (one captured step replayed):
    c3 = configs/mpii-pose.json (v1), 512x512, batch 8 (UNet batch 16), 50-step DDIM, CFG 7.5   (train_...:829-843)
    c5 = mix_lora_and_control_lora.py: v1 ControlLoRA + rank-4 plain LoRA stacked as pre_lora on every processor (:94-121),
         768x768 (96x96 latents), batch 4 (UNet batch 8), 30 steps of DPMSolverMultistepScheduler (:80,153-164)."""
    from controllora_b200.configs import NAMED, wire_processors
    from controllora_b200.sampler import GraphedSampler

    dev = unet.device_
    cl = cb.ControlLoRA.from_config(NAMED["mpii-pose"]).to(dev)
    _randomize_up(torch, cl, dev, 3)
    procs = wire_processors(unet, cl)
    if which == "c5":
        for name, p in procs.items():
            pre = cb.LoRACrossAttnProcessor(p.hidden_size, p.cross_attention_dim, rank=4).to(dev)
            _randomize_up(torch, pre, dev, 5)
            p.inject_pre_lora(pre)
        Bn, size, steps, sched = 4, 768, 30, "dpmpp"
    else:
        Bn, size, steps, sched = 8, 512, 50, "ddim"
    g = torch.Generator().manual_seed(11)
    guide = (torch.rand(Bn, 3, size, size, generator=g) * 2 - 1).to(dev)
    cond = torch.randn(Bn, 77, 768, generator=g).to(dev).to(torch.bfloat16)
    unc = torch.randn(Bn, 77, 768, generator=g).to(dev).to(torch.bfloat16)
    gs = GraphedSampler(unet, cl, Bn, size, size, scheduler=sched, num_inference_steps=steps, guidance_scale=7.5)
    gs(guide, cond, unc, seed=0)                               # warm-up call: hint encoder, capture, full loop
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    lat = gs(guide, cond, unc, seed=1)                         # timed: hint encoder + invariant products + `steps` replays
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return {"value": steps / ms * 1e3, "unit": "denoise steps/s", "ms_total": ms, "steps": steps, "image": size, "batch": Bn,
            "unet_batch": 2 * Bn, "scheduler": sched, "launches_per_step": gs.launches_per_step,
            "latents_finite": bool(torch.isfinite(lat).all()),
            "what": ("configs/mpii-pose.json v1 ControlLoRA, 50-step DDIM + CFG 7.5" if which == "c3" else
                     "mix_lora_and_control_lora.py: v1 ControlLoRA + stacked rank-4 pre-LoRA, 30-step DPM-Solver++(2M) + CFG 7.5") +
                    "; whole call timed (hint encoder + timestep-invariant products once, then one CUDA-graph replay per step)"}


def aux_dropin(torch, cb, unet, config_name, B, steps=4):
    """The path a reference maintainer gets from the import swap alone (INTEGRATION.md): train_...:771-796 verbatim -
    control_lora(guide), unet(...).sample, F.mse_loss, loss.backward() through the autograd bridge, clip_grad_norm_,
    torch.optim.AdamW - no fused Trainer, no CUDA graph."""
    from controllora_b200.configs import NAMED, wire_processors

    dev = unet.device_
    cl = cb.ControlLoRA.from_config(NAMED[config_name]).to(dev)
    _randomize_up(torch, cl, dev, 3)
    wire_processors(unet, cl)
    opt = torch.optim.AdamW(cl.parameters(), lr=1e-4, betas=(0.9, 0.999), weight_decay=1e-2, eps=1e-8)
    x, t, e, guide, tgt = (h.to(dev) for h in synth_inputs(torch, B))
    e = e.to(torch.bfloat16)

    def step():
        cl(guide)
        pred = unet(x, t, e).sample
        loss = torch.nn.functional.mse_loss(pred.float(), tgt.float(), reduction="mean")
        loss.backward()
        torch.nn.utils.clip_grad_norm_(cl.parameters(), 1.0)
        opt.step()
        opt.zero_grad()
        return loss

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / steps * 1e3
    ms = e0.elapsed_time(e1) / steps
    return {"value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "wall_ms_per_step": wall, "steps": steps,
            "final_loss": float(loss), "what": "drop-in classes under torch autograd + torch.optim.AdamW (train_...:771-796 verbatim), "
                                                "per-kernel launches from Python (no fused Trainer, no CUDA graph)"}


def aux_from_pixels(torch, cb, unet, config_name, B, steps=6):
    """The whole loop body train_text_to_image_control_lora.py:751-796 from what the dataloader delivers: pixel_values [B,3,512,512],
    input_ids [B,77], guide [B,3,512,512] -> VAE encode + latent sample (:753-754), CLIP text tower (:768), then the fused step
    (device noise / timesteps / add_noise, hint encoder, UNet fwd / bwd, clip, AdamW; captured CUDA graph).  Frozen SD-1.5-shape VAE
    and text encoder with seeded synthetic weights.  This is the images/s a training run sees once data loading is excluded."""
    from controllora_b200.configs import NAMED, wire_processors
    from controllora_b200.trainer import Trainer

    dev = unet.device_
    cl = cb.ControlLoRA.from_config(NAMED[config_name]).to(dev)
    _randomize_up(torch, cl, dev, 3)
    wire_processors(unet, cl)
    tr = Trainer(unet, cl, lr=1e-4, cuda_graph=True)
    vae = cb.AutoencoderKL.synthetic(dev)
    clip = cb.CLIPTextModel.synthetic(dev)
    g = torch.Generator().manual_seed(7)
    pix = (torch.rand(B, 3, 512, 512, generator=g) * 2 - 1).to(dev)
    ids = torch.randint(0, 49408, (B, 77), generator=g).to(dev)
    guide = (torch.rand(B, 3, 512, 512, generator=g) * 2 - 1).to(dev)
    for _ in range(4):                                   # 2 eager warm-ups, capture, first replay
        loss = tr.step_from_pixels(vae, clip, pix, ids, guide)
    torch.cuda.synchronize()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record()
    for _ in range(steps):
        loss = tr.step_from_pixels(vae, clip, pix, ids, guide)
    e1.record()
    with torch.no_grad():
        for _ in range(steps):
            vae.encode(pix).latent_dist.sample()
            clip(ids)
    e2.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "vae_encode_plus_clip_ms": e1.elapsed_time(e2) / steps, "steps": steps,
            "graph": tr._graph is not None, "final_loss": float(loss),
            "what": "pixels + token ids + guide -> VAE encode + sample, CLIP text tower, fused train step (train_...:751-796 complete); "
                    "synthetic SD-1.5-shape VAE / text-encoder weights"}


def aux_in_child(which, a, timeout_s=240):
    """An auxiliary measurement whose shapes the headline never touches (the 512x512 batch-8 VAE encode) runs in its OWN process: its
    CUDA context, allocator and any failure stay away from the process that has to print the bench line."""
    import subprocess

    cmd = [sys.executable, os.path.abspath(__file__), "--aux-only", which, "--config", a.config, "--batch", str(a.batch)]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s)
    except subprocess.TimeoutExpired:
        return {"value": None, "what": f"child process timed out after {timeout_s} s"}
    for line in reversed(r.stdout.strip().splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    return {"value": None, "what": f"child process failed (rc {r.returncode}): {(r.stderr or r.stdout)[-300:]}"}


def run_aux_only(a):
    try:
        import torch

        import controllora_b200 as cb

        torch.cuda.set_device(0)
        unet = cb.UNet2DConditionModel.synthetic(torch.device("cuda", 0), seed=0)
        out = {"train_from_pixels": lambda: aux_from_pixels(torch, cb, unet, a.config, a.batch)}[a.aux_only]()
    except Exception as ex:
        out = {"value": None, "what": f"failed: {type(ex).__name__}: {ex}"}
    print(json.dumps(out), flush=True)


def aux_gemm_table(torch, ops):
    """Per-shape throughput of the tcgen05 GEMM family at the SD-1.5 shapes (SURVEY 8a census), each timed ALONE with CUDA
    events over operand sets that rotate through > 126 MB (so L2 does not hold them), against the burst bf16 peak of
    MEASURED_PEAKS.json; cuBLAS (torch.matmul) on the same shape is printed beside it for context only."""
    peak = 1667.1
    pth = ROOT / "MEASURED_PEAKS.json"
    if pth.exists():
        peak = json.loads(pth.read_text()).get("bf16_tflops", peak)
    dev = "cuda"
    shapes = [("attn proj + LoRA r4 (north_star)", 32768, 320, 320, True), ("attn proj", 32768, 320, 320, False),
              ("attn proj + LoRA r4", 8192, 640, 640, True), ("attn proj + LoRA r4", 2048, 1280, 1280, True),
              ("ff1", 32768, 2560, 320, False), ("ff2", 32768, 320, 1280, False), ("ff1", 8192, 5120, 640, False),
              ("ff2", 8192, 640, 2560, False), ("ff1", 2048, 10240, 1280, False), ("ff2", 2048, 1280, 5120, False)]
    convs = [(8, 64, 320, 320), (8, 32, 640, 640), (8, 16, 1280, 1280), (8, 64, 640, 320)]
    rows = []

    def timed(fn, nsets, iters=6):
        for i in range(nsets):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            for i in range(nsets):
                fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / (iters * nsets)

    for name, M, N, K, lora in shapes:
        per = 2 * (M * K + M * N)
        nsets = max(2, min(16, int(200e6 // per) + 1))
        As = [torch.randn(M, K, device=dev).to(torch.bfloat16) for _ in range(nsets)]
        Ds = [torch.empty(M, N, device=dev, dtype=torch.bfloat16) for _ in range(nsets)]
        Wt = (torch.randn(N, K, device=dev) / K ** 0.5).to(torch.bfloat16)
        kw = {}
        if lora:
            down = torch.randn(4, K, device=dev) / 4
            kw = dict(ext=ops.split_bf16_ext(down, K), lora_up=torch.randn(N, 4, device=dev) * 0.1, lora_scale=1.0,
                      t_out=torch.empty(M, 4, device=dev))
        ms = timed(lambda i: ops.gemm(As[i], Wt, out=Ds[i], **kw), nsets)
        ms_ref = timed(lambda i: torch.matmul(As[i], Wt.t(), out=Ds[i]), nsets)
        fl = 2.0 * M * N * K + (2.0 * M * 16 * K if lora else 0.0)
        rows.append({"op": name, "M": M, "N": N, "K": K, "lora": lora, "us": ms * 1e3, "tflops": fl / ms / 1e9,
                     "frac_of_burst_peak": fl / ms / 1e9 / peak, "hbm_gbs": (per + 2 * N * K) / ms / 1e6,
                     "cublas_us_no_lora": ms_ref * 1e3, "vs_cublas": ms_ref / ms})
        del As, Ds
    for n, H, Cc, N in convs:
        M, K = n * H * H, 9 * Cc
        per = 2 * (n * H * H * Cc + M * N)
        nsets = max(2, min(16, int(200e6 // per) + 1))
        Xs = [torch.randn(n, H, H, Cc, device=dev).to(torch.bfloat16) for _ in range(nsets)]
        Ds = [torch.empty(n, H, H, N, device=dev, dtype=torch.bfloat16) for _ in range(nsets)]
        Wt = (torch.randn(N, K, device=dev) / K ** 0.5).to(torch.bfloat16)
        ms = timed(lambda i: ops.gemm(Xs[i], Wt, out=Ds[i], conv_stride=1), nsets)
        fl = 2.0 * M * N * K
        rows.append({"op": "conv3x3 (implicit GEMM)", "M": M, "N": N, "K": K, "lora": False, "us": ms * 1e3, "tflops": fl / ms / 1e9,
                     "frac_of_burst_peak": fl / ms / 1e9 / peak, "hbm_gbs": (per + 2 * N * K) / ms / 1e6,
                     "cublas_us_no_lora": None, "vs_cublas": None})
        del Xs, Ds
    return {"rows": rows, "peak_tflops_burst": peak,
            "what": "each shape timed alone (CUDA events, operands rotated through >126 MB); frac = TFLOP/s / measured burst bf16 peak"}


# ------------------------------------------------------------------------------------------------------ GPU arm
DUMP_BUDGET_BYTES = 64_000_000


def dump_outputs(out_dir, tr, loss):
    """What one Trainer.step leaves its caller: the loss, the global gradient norm before clipping, and the trainable parameters
    and AdamW moments after the update, as float32 .npy files under out_dir.  A parameter arena whose three arrays would exceed
    DUMP_BUDGET_BYTES is written as one fixed, seeded sample of its elements: the sorted first k of
    torch.randperm(numel, generator=torch.Generator().manual_seed(0)), the same elements in all three files."""
    import numpy as np
    import torch

    n = tr.numel
    k = min(n, (DUMP_BUDGET_BYTES - 1024) // (3 * 4))        # three float32 arrays; 1 KiB for the two scalars and the .npy headers
    idx = None if k == n else torch.randperm(n, generator=torch.Generator().manual_seed(0))[:k].sort().values.to(tr.flat_p.device)
    arrays = {"loss": loss.reshape(-1), "grad_norm": tr.gnorm_sq.sqrt().reshape(-1) * tr.arena.grad_scale}
    for name, t in (("params", tr.flat_p), ("exp_avg", tr.flat_m), ("exp_avg_sq", tr.flat_v)):
        arrays[name] = t[:n] if idx is None else t[:n][idx]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def run_ours(a):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import controllora_b200 as cb
    from controllora_b200 import _lib, ops
    from controllora_b200.configs import NAMED, wire_processors
    from controllora_b200.trainer import Trainer

    dev = torch.device("cuda", local)
    B = a.batch
    unet = cb.UNet2DConditionModel.synthetic(dev, seed=0)
    torch.manual_seed(0)        # the ControlLoRA's default initialisation: the same weights on every run
    cl = cb.ControlLoRA.from_config(NAMED[a.config]).to(dev)
    g = torch.Generator().manual_seed(3)
    with torch.no_grad():       # LoRA `up` weights are zero-initialised: give them values so no path is trivially dead
        for n_, p_ in cl.named_parameters():
            if n_.endswith("up.weight"):
                p_.copy_((0.02 * torch.randn(p_.shape, generator=g)).to(dev))
    wire_processors(unet, cl)
    tr = Trainer(unet, cl, lr=1e-4, cuda_graph=not a.no_graph)   # fwd/bwd captured once, replayed every step
    host = synth_inputs(torch, B, seed_off=rank)
    x, t, e, guide, tgt = (h.to(dev) for h in host)
    e = e.to(torch.bfloat16)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def trace(msg):           # CLB_BENCH_TRACE=1: per-rank phase markers on stderr (to locate a multi-rank stall)
        if os.environ.get("CLB_BENCH_TRACE"):
            print(f"[bench rank {rank}] {msg}", file=sys.stderr, flush=True)

    trace("warm-up")
    for _ in range(max(a.warmup, 3)):
        loss = tr.step(x, t, e, guide, tgt)
    barrier()
    trace("timed region")
    # ---------------- timed region: inputs resident in HBM
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(a.steps):
        loss = tr.step(x, t, e, guide, tgt)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, tr, loss)      # before the end-to-end and roofline passes below train further
    launches = (_lib.launch_count() - n0) // max(a.steps, 1)
    if tr.cuda_graph and tr.launches_per_step:
        launches = tr.launches_per_step      # kernels inside the replayed graph (counted at capture) + optimizer launches
    clocks = sampler.stop() if rank == 0 else None
    tmax = torch.tensor([ms_total], device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_step = float(tmax) / a.steps
    value = world * B / (ms_step / 1e3)
    final_loss = float(loss)
    # data-parallel sanity: every rank trained on its own batch, so the replicas are in sync only if the gradient exchange works
    replicas_in_sync = None
    if world > 1:
        chk = torch.stack([tr.flat_p.double().sum(), (tr.flat_p.double() ** 2).sum()])
        allc = [torch.empty_like(chk) for _ in range(world)]
        dist.all_gather(allc, chk)
        replicas_in_sync = bool(all(torch.equal(allc[0], c) for c in allc[1:]))

    trace("end-to-end region")
    # ---------------- end-to-end: host (pinned) buffers in, loss out, every step
    pinned = [h.pin_memory() for h in host]
    h2d = sum(p.numel() * p.element_size() for p in pinned)
    # two device staging sets: the copy stream uploads step i+1 while the compute stream runs step i (what a training loop
    # with a prefetching loader does); every step still moves all of its inputs host->device and its loss device->host
    dbuf = [[torch.empty_like(p, device=dev) for p in pinned] for _ in range(2)]
    loss_host = torch.empty(1, dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def prefetch(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])          # the step that last read this slot has finished with it
            for d, p in zip(dbuf[slot], pinned):
                d.copy_(p, non_blocking=True)
            ready[slot].record(copy_stream)

    def e2e_run(nsteps):
        cur = torch.cuda.current_stream()
        for ev in consumed:
            ev.record(cur)
        prefetch(0)
        last = None
        for i in range(nsteps):
            slot = i & 1
            cur.wait_event(ready[slot])
            if i + 1 < nsteps:
                prefetch(slot ^ 1)
            d = dbuf[slot]
            l = tr.step(d[0], d[1], ops.f32_to_bf16(d[2]), d[3], d[4])
            consumed[slot].record(cur)
            loss_host.copy_(l, non_blocking=True)
            cur.synchronize()
            last = float(loss_host)
        return last

    e2e_run(2)
    barrier()
    t0 = time.perf_counter()
    e2e_run(a.steps)
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = world * B * a.steps / float(dt)

    # ---------------- roofline of the dominant kernel family (tcgen05 GEMM / implicit-GEMM conv): live CUDA-event timing
    trace("roofline passes")
    roof = None
    if world > 1 and not a.no_roofline:
        # the eager passes below contain the gradient all-reduce: every rank has to run them (only rank 0 keeps the timings)
        barrier()
    if not a.no_roofline:
        peak_tf, peak_hbm, which = measured_peaks()
        rec = []
        orig = ops.gemm

        def timed_gemm(A_, B_, **kw):
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            r = orig(A_, B_, **kw)
            s1.record()
            conv = kw.get("conv_stride", 0)
            M = A_.shape[0] if not conv else A_.shape[0] * A_.shape[1] * A_.shape[2] // (conv * conv)
            N, K = B_.shape
            fl = 2.0 * M * N * K + (2.0 * M * 16 * K if kw.get("lora_up") is not None else 0.0)
            # algorithmic bytes of the launch: A, W and D once each in their storage type (+ the residual read when fused)
            by = 2.0 * (A_.numel() + N * K) + (4.0 if kw.get("out_fp32") else 2.0) * M * N + (2.0 * M * N if kw.get("residual") is not None else 0.0)
            rec.append((fl, s0, s1, by))
            return r

        ops.gemm = timed_gemm
        import controllora_b200.engine as E_, controllora_b200.lora_runtime as LR_, controllora_b200.hint_encoder as HE_
        # uncaptured passes so that every GEMM launch can be bracketed by events; the first one only re-warms the caching
        # allocator (the graph capture emptied it), the second one is measured
        tr.step(x, t, e, guide, tgt, eager=True)
        torch.cuda.synchronize()
        rec.clear()
        tr.step(x, t, e, guide, tgt, eager=True)
        torch.cuda.synchronize()
        ops.gemm = orig
        fl = sum(r[0] for r in rec)
        tm = sum(r[1].elapsed_time(r[2]) for r in rec)
        alg_bytes = sum(r[3] for r in rec)
        ach = fl / (tm * 1e-3) / 1e12
    if rank == 0 and not a.no_roofline:
        roof = {"bound": "tensor", "kernel": "gemm_tc_kernel<BN,EXT,BK> (all fused linear / LoRA / implicit-GEMM conv launches of one step)",
                "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf, "traffic": gemm_traffic_per_launch(),
                "launches_per_step": len(rec), "gemm_ms_per_step": tm, "algorithmic_gflop_per_step": fl / 1e9,
                "algorithmic_bytes_per_step": alg_bytes, "algorithmic_bytes_per_launch": alg_bytes / max(len(rec), 1),
                "peak_source": which,
                "step_model_flops_utilisation": (GFLOP_PER_IMAGE_STEP * 1e9 * B / (ms_step * 1e-3)) / (peak_tf * 1e12)}
    # ---------------- auxiliary numbers (rank 0, after every measurement of the headline): BASELINE configs C3 / C5 denoise
    #                  steps/s, the drop-in (autograd + torch.optim.AdamW) path, and the per-shape GEMM table
    trace("aux")
    aux = {}
    graph_used = bool(tr.cuda_graph and tr._graph is not None)
    if rank == 0 and world == 1 and not a.no_aux:      # single-GPU numbers: a scaling run must not keep N-1 ranks waiting on them
        del tr
        torch.cuda.empty_cache()
        for key, fn in (("denoise_c3", lambda: aux_denoise(torch, cb, unet, "c3")), ("denoise_c5", lambda: aux_denoise(torch, cb, unet, "c5")),
                        ("dropin_train_step", lambda: aux_dropin(torch, cb, unet, a.config, B)),
                        ("train_from_pixels", lambda: aux_in_child("train_from_pixels", a)),
                        ("gemm_per_shape", lambda: aux_gemm_table(torch, ops))):
            try:
                aux[key] = fn()
            except Exception as ex:      # an auxiliary number must never take the headline down
                aux[key] = {"value": None, "what": f"failed: {type(ex).__name__}: {ex}"}
            torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
    trace("report")

    if rank == 0:
        cpu = None
        if world == 1 and not a.no_cpu_baseline:
            try:
                cpu = cpu_baseline(a.config)
            except Exception as ex:  # the baseline must never take the measurement down
                cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": f"{a.config} ControlLoRA train step on the SD-1.5 UNet, 512x512 (64x64 latents, 77x768 text states), "
                                   f"batch {B}/GPU, hint encoder + UNet fwd/bwd + clip + AdamW" + (" + NCCL all-reduce of the flat grad arena" if world > 1 else ""),
                       "global_batch": world * B, "parallelism": f"dp{world}", "replicas_in_sync": replicas_in_sync,
                       "cuda_graph": graph_used,
                       "l2_policy": "no explicit flush: each step streams 1.7 GB of frozen weights plus >5 GB of activations, far beyond the 126 MB L2",
                       "weights": "random-init (seeded), SD-1.5 / ControlLoRA shapes", "final_loss": final_loss},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if roof is not None:
            out["roofline"] = roof
        if aux:
            out["aux"] = aux
            if roof is not None and isinstance(aux.get("gemm_per_shape"), dict) and aux["gemm_per_shape"].get("rows"):
                roof["per_shape"] = aux["gemm_per_shape"]["rows"]
        if cpu is not None:
            out["cpu_baseline"] = cpu
        print(json.dumps(out), flush=True)
    if world > 1:
        # orderly teardown, then a hard exit: a rank must never linger in NCCL / CUDA-graph destructors after the line is out
        trace("teardown")
        try:
            tr._graph = None
        except NameError:
            pass
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    a = parse()
    if a.aux_only:
        run_aux_only(a)
        return
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
