"""Inference with the CNN's maps in f32 against fp16 / bf16 (CUDA autocast), timed with CUDA events.

    python scripts/autocast_infer_bench.py [--iters 20] [--warmup 3]

Part 1, the fused Retinex + CLAHE call alone (native.retinex_clahe / retinex_clahe_u8) at 64 x 1080p with the map pairs
(illu, e) = (f32, f32), (f32, fp16) -- what the real network emits under autocast -- and (fp16, fp16), alternating call by call.
Bytes per pixel are the frames the call streams: x 12 + illu s_i + e 3 s_e read, the f32 frame 12 or the u8 frame 3 written
(the 3 B/px u8 Lab intermediate, written once and re-read from L2 / HBM, is left out as in DESIGN.md §1).

Part 2, the batch driver's device work end to end: enhance_frames_u8 with UP_Retinex (random weights) at 8 x 1080p, under no
autocast, fp16 and bf16 autocast -- the CNN plus the fused u8 call.

Prints one JSON line per case, and the card's name and power limit.  Every working set of part 1 exceeds the 126 MB L2."""
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

from retinex_image_enhancement_b200 import native  # noqa: E402

PAIRS = [(torch.float32, torch.float32), (torch.float32, torch.float16), (torch.float16, torch.float16)]


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except Exception:
        power = "unknown"
    return name, power


def bytes_per_px(di, de, u8):
    return 12 + torch.finfo(di).bits // 8 + 3 * (torch.finfo(de).bits // 8) + (3 if u8 else 12)


def time_arms(arms, iters, warmup):
    """{name: median ms} of the callables in `arms`, run alternately."""
    for fn in arms.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(iters):
        for k, fn in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            times[k].append(a.elapsed_time(b))
    return {k: statistics.median(v) for k, v in times.items()}


def part1(args, name, power):
    n, h, w = 64, 1080, 1920
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.rand((n, 3, h, w), device="cuda", generator=g)
    illu32 = torch.rand((n, 1, h, w), device="cuda", generator=g) * 0.9 + 0.05
    e32 = torch.rand((n, 3, h, w), device="cuda", generator=g)
    ops = {di_de: (illu32.to(di_de[0]), e32.to(di_de[1])) for di_de in PAIRS}
    for u8 in (False, True):
        fn = native.retinex_clahe_u8 if u8 else native.retinex_clahe
        outs = {k: fn(x, il, e, autocast=True) for k, (il, e) in ops.items()}
        arms = {k: (lambda il=il, e=e, o=outs[k]: fn(x, il, e, out=o, autocast=True)) for k, (il, e) in ops.items()}
        ms = time_arms(arms, args.iters, args.warmup)
        base = ms[PAIRS[0]]
        for (di, de), t in ms.items():
            bpp = bytes_per_px(di, de, u8)
            print(json.dumps({
                "part": "retinex_clahe_u8" if u8 else "retinex_clahe", "shape": [n, 3, h, w],
                "illu": str(di)[6:], "e": str(de)[6:], "bytes_per_px": bpp, "ms": round(t, 3),
                "vs_f32_maps": round(base / t, 3), "rate_tb_s": round(bpp * n * h * w / (t / 1e3) / 1e12, 2),
                "card": name, "power_limit": power}))
        del outs, arms
    del x, illu32, e32, ops
    torch.cuda.empty_cache()


def part2(args, name, power):
    from retinex_image_enhancement_b200.enhancers.simple_enhance import amp_context, enhance_frames_u8
    from retinex_image_enhancement_b200.models.model import UP_Retinex
    torch.manual_seed(0)
    model = UP_Retinex().cuda().eval()
    low = torch.rand((8, 3, 1080, 1920), device="cuda")

    def run(amp):
        with amp_context(amp):
            return enhance_frames_u8(model, low)

    ms = time_arms({amp: (lambda amp=amp: run(amp)) for amp in (None, "fp16", "bf16")}, max(args.iters // 4, 3), args.warmup)
    for amp, t in ms.items():
        print(json.dumps({"part": "enhance_frames_u8 UP_Retinex", "shape": [8, 3, 1080, 1920], "amp": amp or "off",
                          "ms": round(t, 2), "vs_f32": round(ms[None] / t, 3), "card": name, "power_limit": power}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("autocast_infer_bench: needs a CUDA device")
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power}))
    with torch.no_grad():
        part1(args, name, power)
        part2(args, name, power)


if __name__ == "__main__":
    main()
