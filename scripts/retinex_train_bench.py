"""Forward + backward of the two Retinex lines of a training step (models/model.py:405-413, :442) under autograd: the stock torch
expressions against the fused kernels (models.model._RetinexFn), alternating step by step in one run, timed with CUDA events.

    python scripts/retinex_train_bench.py [--iters 20] [--warmup 3] [--step-iters 10]

Each step: R, enhanced = f(x, illu, e) with illu and e requiring a gradient (the CNN's outputs), then the gradients of illu and e
from upstream gradients on both outputs.  Map pairs (illu, e): f32 / f32; fp16 / fp16 under fp16 autocast; and f32 / fp16,
f32 / bf16 under fp16 / bf16 autocast, the pair the real network emits there (its illumination head adds the f32 mean(x)).
Prints one JSON line per (shape, maps) and the card's name and power limit.  Algorithmic bytes are those of the fused path:
forward x 12 + illu si + e 3se read, R 12 + enhanced 12 written; backward g_enh 12 + g_refl 12 + x 12 + illu si + e 3se read,
g_illu si + g_e 3se written (si / se = bytes of an illu / e element): 120 B/px in f32, 96 in fp16, 102 for f32 / fp16.  Every
working set below is larger than the 126 MB L2, so each pass streams from HBM; the script states it per shape.

Then one whole UP_Retinex training step at the trainer's 8x3x640^2 under fp16 autocast with a GradScaler (forward, a simple
L1 + mean loss, scaled backward, Adam step, scale update), the Retinex lines on the stock expressions against the fused kernels,
alternating step by step, with the peak memory of one step.  The loss stands in for the trainer's criterion, whose decoupling,
perceptual and frequency terms are stock torch either way."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from retinex_image_enhancement_b200.models import model as M  # noqa: E402

SHAPES = [(8, 640, 640), (32, 640, 640), (16, 1080, 1920)]   # trainer default, a large batch, 1080p frames
L2_BYTES = 126e6
HBM_PEAK = 7.7e12   # B/s, HGX B200 data sheet, one GPU at up to 1000 W


def stock(x, illu, e):
    r = x / (illu + M.EPSILON)
    return r, r * e + (1 - r) * (e ** 2)


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except Exception:
        power = "unknown"
    return name, power


# (illu dtype, e dtype, autocast dtype or None)
PAIRS = [(torch.float32, torch.float32, None), (torch.float16, torch.float16, torch.float16),
         (torch.float32, torch.float16, torch.float16), (torch.float32, torch.bfloat16, torch.bfloat16)]


def bytes_per_px(si, se):
    return (12 + si + 3 * se + 12 + 12) + (12 + 12 + 12 + si + 3 * se + si + 3 * se)


def timed_arms(arms, step, iters, warmup):
    """Median CUDA-event time of step(arm) per arm, the arms alternating, and the peak memory of one step above what was
    allocated before it."""
    times = {k: [] for k in arms}
    peaks = {}
    for k, fn in arms.items():
        for _ in range(warmup):
            step(fn)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        step(fn)
        torch.cuda.synchronize()
        peaks[k] = torch.cuda.max_memory_allocated() - base
    for _ in range(iters):
        for k, fn in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step(fn)
            b.record()
            b.synchronize()
            times[k].append(a.elapsed_time(b))
    return {k: statistics.median(v) for k, v in times.items()}, peaks


def training_step(args, name, power):
    """One UP_Retinex training step under fp16 autocast + GradScaler at 8x3x640^2, stock Retinex lines against fused."""
    dev = torch.device("cuda")
    torch.manual_seed(0)
    model = M.UP_Retinex().to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    scaler = torch.amp.GradScaler("cuda")
    gen = torch.Generator(device=dev).manual_seed(1)
    x = torch.rand((8, 3, 640, 640), device=dev, generator=gen)
    target = torch.rand((8, 3, 640, 640), device=dev, generator=gen)
    fused_autograd = M._fused_autograd

    def step(fused):
        M._fused_autograd = fused_autograd if fused else (lambda *a: False)
        try:
            opt.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.float16):
                enh, r, _ = model(x)
                loss = (enh - target).abs().mean() + 0.1 * r.mean()
            scaler.scale(loss).backward()
            scaler.step(opt)
            scaler.update()
        finally:
            M._fused_autograd = fused_autograd

    ms, peaks = timed_arms({"stock": False, "fused": True}, step, args.step_iters, args.warmup)
    print(json.dumps({
        "training_step": [8, 3, 640, 640], "autocast": "float16", "grad_scaler": True,
        "stock_ms": round(ms["stock"], 2), "fused_ms": round(ms["fused"], 2), "speedup": round(ms["stock"] / ms["fused"], 3),
        "peak_alloc_mb": {k: round(v / 1e6, 1) for k, v in peaks.items()}, "card": name, "power_limit": power}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--step-iters", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("retinex_train_bench: needs a CUDA device")
    dev = torch.device("cuda")
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power}))
    for (n, h, w), (illu_dt, e_dt, amp) in [(s, p) for s in SHAPES for p in PAIRS]:
        si, se = torch.empty((), dtype=illu_dt).element_size(), torch.empty((), dtype=e_dt).element_size()
        gen = torch.Generator(device=dev).manual_seed(n * h)
        x = torch.rand((n, 3, h, w), device=dev, generator=gen)
        illu = (torch.rand((n, 1, h, w), device=dev, generator=gen) * 0.9 + 0.05).to(illu_dt).requires_grad_()
        e = torch.rand((n, 3, h, w), device=dev, generator=gen).to(e_dt).requires_grad_()
        g_refl, g_enh = torch.rand_like(x) - 0.5, torch.rand_like(x) - 0.5
        px = n * h * w
        working_set = px * (12 + si + 3 * se + 12 + 12 + 12 + 12 + si + 3 * se)   # every tensor the step touches, once

        def step(fn):
            with torch.autocast("cuda", dtype=amp or torch.float16, enabled=amp is not None):
                r, enh = fn(x, illu, e)
            return torch.autograd.grad([r, enh], [illu, e], [g_refl, g_enh])

        ms, peaks = timed_arms({"stock": stock, "fused": M.retinex_recombine}, step, args.iters, args.warmup)
        alg = bytes_per_px(si, se) * px
        print(json.dumps({
            "shape": [n, 3, h, w], "maps": [str(illu_dt).replace("torch.", ""), str(e_dt).replace("torch.", "")],
            "autocast": str(amp).replace("torch.", "") if amp else False,
            "working_set_mb": round(working_set / 1e6, 1), "fits_l2": working_set <= L2_BYTES,
            "stock_ms": round(ms["stock"], 3), "fused_ms": round(ms["fused"], 3), "speedup": round(ms["stock"] / ms["fused"], 2),
            "algorithmic_bytes_per_px": bytes_per_px(si, se),
            "fused_rate_tb_s": round(alg / (ms["fused"] / 1e3) / 1e12, 2),
            "fused_frac_of_7p7": round(alg / (ms["fused"] / 1e3) / HBM_PEAK, 3),
            "peak_alloc_mb": {k: round(v / 1e6, 1) for k, v in peaks.items()},
            "card": name, "power_limit": power}))
        del x, illu, e, g_refl, g_enh
        torch.cuda.empty_cache()
    training_step(args, name, power)


if __name__ == "__main__":
    main()
