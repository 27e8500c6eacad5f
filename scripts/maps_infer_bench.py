"""Content-aware, multi-scale and predict inference from the CNN maps: the fused map epilogues against the composition the drivers
ran before (recombination writing R and enhanced, then the mode's passes, then the u8 quantiser), timed with CUDA events.

    python scripts/maps_infer_bench.py [--iters 15] [--warmup 3]

Part 1, the device stage alone at 64 x 1080p and 16 x 4K with the map pairs (illu, e) = (f32, f32) and (f32, fp16), for the
f32 results (content-aware, multi-scale) and the stored u8 pair (content-aware, multi-scale, predict), composition and fused
alternating call by call.  bytes_per_px are the algorithmic bytes of each arm counted from shapes (DESIGN.md §7); peak_mb is
torch.cuda.max_memory_allocated during one call of the arm, above what was allocated before it.

Part 2, the driver's device side end to end: enhance_frames_host_u8 in content-aware and in multi-scale mode at 64 x 1080p
with a pointwise stub CNN, once with forward_maps (the fused path) and once with it hidden (model(x)).

Prints one JSON line per case, and the card's name and power limit.  Every working set exceeds the 126 MB L2."""
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

PAIRS = [(torch.float32, torch.float32), (torch.float32, torch.float16)]
MODES = ["ca", "ms", "ca8", "ms8", "pred8"]


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except Exception:
        power = "unknown"
    return name, power


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


def bytes_per_px(mode, fused, si, se):
    """Algorithmic bytes per pixel: x 12, illu si, e 3 se, f32 frames 12, planes 4, u8 frames 3 + 1."""
    maps = 12 + si + 3 * se
    u8 = mode.endswith("8")
    if not fused:
        recombine = maps + 24                                  # R and enhanced written
        tail = 20 if u8 else 0                                 # quantise enhanced (12 + 3) and illu (4 + 1)
        body = {"ca": 60, "ms": 36, "pr": 0}[mode[:2]]         # the mode's passes over x and enhanced
        return recombine + body + tail
    if mode.startswith("ca"):                                 # blur pass, attention pass, epilogue
        return (16 + 20 + 4 + maps + 4) if u8 else (20 + 12 + 4 + maps + 12)
    if mode.startswith("ms"):                                 # statistics pass, epilogue
        return 12 + maps + (4 if u8 else 12)
    return maps + 4


def composition(mode, x, illu, e):
    _, enh = native.retinex_recombine_typed(x, illu, e, autocast=True)
    if mode.startswith("ca"):
        out = native.content_aware_apply(x, enh, out=enh)
    elif mode.startswith("ms"):
        out = native.multiscale_enhance(x, enh, out=enh)[0]
    else:
        out = enh
    if mode.endswith("8"):
        return native.quantize_u8(out), native.quantize_u8(illu.float().contiguous())
    return out


def fused(mode, x, illu, e):
    fn = {"ca": native.retinex_content_aware, "ca8": native.retinex_content_aware_u8, "ms": native.retinex_multiscale,
          "ms8": native.retinex_multiscale_u8, "pred8": native.retinex_quantize_u8}[mode]
    return fn(x, illu, e, autocast=True)


def peak_mb(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    r = fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    del r
    return round(peak / 2 ** 20, 1)


def part1(args, name, power):
    for n, h, w in ((64, 1080, 1920), (16, 2160, 3840)):
        g = torch.Generator(device="cuda").manual_seed(1)
        x = torch.rand((n, 3, h, w), device="cuda", generator=g)
        illu32 = torch.rand((n, 1, h, w), device="cuda", generator=g) * 0.9 + 0.05
        e32 = torch.rand((n, 3, h, w), device="cuda", generator=g) * 1.2
        for di, de in PAIRS:
            illu, e = illu32.to(di), e32.to(de)
            si, se = torch.finfo(di).bits // 8, torch.finfo(de).bits // 8
            for mode in MODES:
                if mode in ("ca", "ms"):
                    torch.cuda.empty_cache()
                arms = {"composition": lambda: composition(mode, x, illu, e), "fused": lambda: fused(mode, x, illu, e)}
                got, want = arms["fused"](), arms["composition"]()
                same = all(torch.equal(a, b) for a, b in zip(got if isinstance(got, tuple) else (got,),
                                                             want if isinstance(want, tuple) else (want,)))
                del got, want
                peaks = {k: peak_mb(fn) for k, fn in arms.items()}
                ms = time_arms(arms, args.iters, args.warmup)
                for arm, t in ms.items():
                    bpp = bytes_per_px(mode, arm == "fused", si, se)
                    print(json.dumps({
                        "part": "device", "mode": mode, "arm": arm, "shape": [n, 3, h, w], "illu": str(di)[6:], "e": str(de)[6:],
                        "bytes_per_px": bpp, "ms": round(t, 3), "rate_tb_s": round(bpp * n * h * w / (t / 1e3) / 1e12, 2),
                        "speedup": round(ms["composition"] / t, 3), "peak_mb": peaks[arm], "bit_equal": same,
                        "card": name, "power_limit": power}), flush=True)
            del illu, e
        del x, illu32, e32
        torch.cuda.empty_cache()


class StubCNN(torch.nn.Module):
    """A pointwise stand-in for the CNN: the real network's time would hide the stage this part measures."""

    def forward_maps(self, x):
        return x.mean(dim=1, keepdim=True) * 0.5 + 0.25, torch.sqrt(x)

    def forward(self, x):
        from retinex_image_enhancement_b200.models.model import retinex_recombine
        illu, e = self.forward_maps(x)
        reflectance, enhanced = retinex_recombine(x.contiguous(), illu.contiguous(), e.contiguous())
        return enhanced, reflectance, illu


class Hidden(torch.nn.Module):
    def __init__(self, inner):
        super().__init__()
        self.inner = inner

    def forward(self, x):
        return self.inner(x)


def part2(args, name, power):
    from retinex_image_enhancement_b200.enhancers.simple_enhance import enhance_frames_host_u8
    n, h, w = 64, 1080, 1920
    frames = torch.randint(0, 90, (n, h, w, 3), dtype=torch.uint8).pin_memory()
    stub = StubCNN().eval()
    models = {"fused": stub, "composition": Hidden(stub).eval()}
    for ca in (True, False):
        outs = {k: (torch.empty((n, h, w, 3), dtype=torch.uint8).pin_memory(), torch.empty((n, h, w, 1), dtype=torch.uint8).pin_memory())
                for k in models}

        def step(k):
            for ev in enhance_frames_host_u8(models[k], frames, outs[k][0], outs[k][1], "cuda", enable_content_aware=ca,
                                             enable_multi_scale=not ca, chunk=8):
                ev.synchronize()

        ms = time_arms({k: (lambda k=k: step(k)) for k in models}, max(args.iters // 3, 3), args.warmup)
        same = all(torch.equal(a, b) for a, b in zip(outs["fused"], outs["composition"]))
        for arm, t in ms.items():
            print(json.dumps({"part": "enhance_frames_host_u8", "mode": "content_aware" if ca else "multi_scale", "arm": arm,
                              "shape": [n, h, w, 3], "ms": round(t, 2), "mpix_s": round(n * h * w / 1e6 / (t / 1e3), 1),
                              "speedup": round(ms["composition"] / t, 3), "bit_equal": same, "card": name,
                              "power_limit": power}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("maps_infer_bench: needs a CUDA device")
    name, power = card()
    print(json.dumps({"card": name, "power_limit": power}), flush=True)
    with torch.no_grad():
        part1(args, name, power)
        part2(args, name, power)


if __name__ == "__main__":
    main()
