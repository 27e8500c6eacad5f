"""Forward + backward of the two Retinex lines of a training step (models/model.py:405-413, :442) under autograd: the stock torch
expressions against the fused kernels (models.model._RetinexFn), alternating step by step in one run, timed with CUDA events.

    python scripts/retinex_train_bench.py [--iters 20] [--warmup 3]

Each step: R, enhanced = f(x, illu, e) with illu and e requiring a gradient (the CNN's outputs), then the gradients of illu and e
from upstream gradients on both outputs.  Maps are f32, or fp16 under autocast (what the CNN emits there).  Prints one JSON line
per (shape, mode) and the card's name and power limit.  Algorithmic bytes are those of the fused path: forward x 12 + illu s +
e 3s read, R 12 + enhanced 12 written; backward g_enh 12 + g_refl 12 + x 12 + illu s + e 3s read, g_illu s + g_e 3s written
(s = bytes of a map element): 120 B/px in f32, 96 in fp16.  Every working set below is larger than the 126 MB L2, so each pass
streams from HBM; the script states it per shape."""
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


def bytes_per_px(s):
    return (12 + s + 3 * s + 12 + 12) + (12 + 12 + 12 + s + 3 * s + s + 3 * s)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("retinex_train_bench: needs a CUDA device")
    dev = torch.device("cuda")
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power}))
    for (n, h, w), amp in [(s, a) for s in SHAPES for a in (False, True)]:
        dt = torch.float16 if amp else torch.float32
        s = 2 if amp else 4
        gen = torch.Generator(device=dev).manual_seed(n * h)
        x = torch.rand((n, 3, h, w), device=dev, generator=gen)
        illu = (torch.rand((n, 1, h, w), device=dev, generator=gen) * 0.9 + 0.05).to(dt).requires_grad_()
        e = torch.rand((n, 3, h, w), device=dev, generator=gen).to(dt).requires_grad_()
        g_refl, g_enh = torch.rand_like(x) - 0.5, torch.rand_like(x) - 0.5
        px = n * h * w
        working_set = px * (12 + s + 3 * s + 12 + 12 + 12 + 12 + s + 3 * s)   # every tensor the step touches, once

        def step(fn):
            with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
                r, enh = fn(x, illu, e)
            return torch.autograd.grad([r, enh], [illu, e], [g_refl, g_enh])

        arms = {"stock": stock, "fused": M.retinex_recombine}
        times = {k: [] for k in arms}
        peaks = {}
        for k, fn in arms.items():
            for _ in range(args.warmup):
                step(fn)
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            step(fn)
            torch.cuda.synchronize()
            peaks[k] = torch.cuda.max_memory_allocated() - base
        for _ in range(args.iters):
            for k, fn in arms.items():
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                step(fn)
                b.record()
                b.synchronize()
                times[k].append(a.elapsed_time(b))
        ms = {k: statistics.median(v) for k, v in times.items()}
        alg = bytes_per_px(s) * px
        print(json.dumps({
            "shape": [n, 3, h, w], "maps": str(dt).replace("torch.", ""), "autocast": amp,
            "working_set_mb": round(working_set / 1e6, 1), "fits_l2": working_set <= L2_BYTES,
            "stock_ms": round(ms["stock"], 3), "fused_ms": round(ms["fused"], 3), "speedup": round(ms["stock"] / ms["fused"], 2),
            "algorithmic_bytes_per_px": bytes_per_px(s),
            "fused_rate_tb_s": round(alg / (ms["fused"] / 1e3) / 1e12, 2),
            "fused_frac_of_7p7": round(alg / (ms["fused"] / 1e3) / HBM_PEAK, 3),
            "peak_alloc_mb": {k: round(v / 1e6, 1) for k, v in peaks.items()},
            "card": name, "power_limit": power}))
        del x, illu, e, g_refl, g_enh
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
