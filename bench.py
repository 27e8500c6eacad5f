#!/usr/bin/env python3
"""bench.py -- the headline benchmark of upretinex-b200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2|c3|c4|c5] [--no-named]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Metric (BASELINE.json): Mpix/s of the 1080p CLAHE+Retinex enhance path.  Default workload "c2" = BASELINE
config 2: a batch of 64 synthetic 1920x1080 f32 RGB frames per GPU through the CLAHE-in-Lab op
(upr_clahe_lab_f32, SURVEY section 8d: 24 algorithmic bytes per pixel).  One step = one pass of the op over the
whole batch.  Frames are independent, so N GPUs each own their own 64 frames (weak scaling, no collective).

  value      device-resident inputs, CUDA-event timed, max over ranks
  e2e        same op through the reference-facing Python API with HOST tensors in and out
             (AdaptiveParameterAdjuster.apply_clahe_enhancement -> upr_clahe_lab_f32_host): the pinned host ->
             device copy of every frame and the device -> host copy of every result are inside the timed region
  e2e_driver the enhance DRIVER's own boundary (enhancers/simple_enhance.py): host uint8 frames as decoded from files in,
             host uint8 frames as save_image stores them out (3 B/px up, 3 + 1 B/px down), Retinex recombination + CLAHE
             fused on the device (CNN stubbed: out of scope)
  roofline   dominant kernel's algorithmic bytes / its CUDA-event duration vs MEASURED_PEAKS.json hbm_gbs
  named_configs  the other BASELINE configs as sub-records, each with its own roofline and clocks, at the GPU count of the run:
             c3 256 4K frames over the N GPUs (multi-scale statistics + gain), c4 texture statistics + all-reduce of the batch
             statistics (NCCL vs the fused peer-memory kernel, bit-equality flag), c5 128 4K frames per GPU in chunks of 16
             through content-aware + multi-scale with one shared epilogue
  cpu_baseline / --impl reference
             the reference's CPU path on the host cores: the UNMODIFIED reference class when its tree is present
             (UPR_REFERENCE, baseline/_ref, /root/reference), else the restatement of its call sequence
             (oracle/cv2_chain.py); the restatement on a thread pool over frames is reported beside it
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Mpix/s, 1080p CLAHE+Retinex enhance"
UNIT = "Mpix/s"
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback ("of fallback")
C2_FRAMES, C2_H, C2_W = 64, 1080, 1920
C2_CONFIG = {"workload": "c2: CLAHE-in-Lab (upr_clahe_lab_f32 / adaptive_params.py:121-169, clip 2.0, 8x8 tiles) over 64 synthetic "
                         "1920x1080 f32 RGB frames per GPU (BASELINE config 2)", "frames_per_gpu": C2_FRAMES, "h": C2_H, "w": C2_W,
             "l2": "inputs larger than L2 (1.59 GB read + 1.59 GB written per step vs 126 MB L2), no flush needed",
             "sharding": "by frame, no collective"}


# ---------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------
def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int, period_s: float = 0.004):
        self.samples, self.reasons, self.max_mhz, self.err = [], set(), None, None
        self._stop = threading.Event()
        self._thread = None
        self.period = period_s
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # pragma: no cover
            self.nv, self.err = None, repr(e)

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception as e:  # pragma: no cover
                self.err = repr(e)
                return
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0,
                    "note": self.err or "no samples"}
        return {"sm_mhz": int(statistics.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def make_frames(torch, n, h, w, seed, device):
    """Synthetic batch of SURVEY section 8d: 50 % dark (0.3*U), 25 % uniform, 25 % ramp / constant 0.3."""
    g = torch.Generator(device=device).manual_seed(seed)
    x = torch.rand((n, 3, h, w), device=device, generator=g)
    for i in range(n):
        k = i % 4
        if k in (0, 2):
            x[i] *= 0.3
        elif k == 3:
            if (i // 4) % 2 == 0:
                x[i] = 0.3
            else:
                xs = torch.linspace(0, 1, w, device=device)[None, :].expand(h, w)
                ys = torch.linspace(0, 1, h, device=device)[:, None].expand(h, w)
                x[i, 0], x[i, 1], x[i, 2] = xs, ys, (xs + ys) / 2
    return x


DUMP_BYTES = 48 << 20   # --dump-outputs: the files of one run stay well under 64 MB in all


def dump_outputs(dirname, arrays):
    """Write the arrays the timed path returned in its last step as DIR/<name>.npy (float32).  Arrays up to 1 MB are written
    whole; a larger [N,C,H,W] output is reduced to a fixed, seeded sample (the same image rows of the same frames on every
    run), so that two builds of the project can be compared output for output.  Everything written fits in DUMP_BYTES."""
    import numpy as np
    import torch
    big = [k for k, t in arrays.items() if t.numel() * 4 > (1 << 20)]
    small = sum(t.numel() * 4 for k, t in arrays.items() if k not in big)
    if small > DUMP_BYTES or any(arrays[k].dim() != 4 for k in big):
        raise ValueError("--dump-outputs samples one [N,C,H,W] output per name; these arrays do not fit its budget")
    share = (DUMP_BYTES - small) // max(1, len(big))
    os.makedirs(dirname, exist_ok=True)
    written = 0
    for name, t in arrays.items():
        t = t.detach().float()
        if name in big:
            n, c, h, w = t.shape
            rng = np.random.default_rng(0)
            row_bytes = c * w * 4
            frames = min(n, max(1, share // row_bytes))
            rows = min(h, max(1, share // (frames * row_bytes)))
            ri = torch.from_numpy(np.sort(rng.choice(h, rows, replace=False))).to(t.device)
            fi = torch.from_numpy(np.sort(rng.choice(n, frames, replace=False))).to(t.device)
            t = t.index_select(2, ri).index_select(0, fi)
        a = t.cpu().numpy()
        written += a.nbytes
        if written > DUMP_BYTES:
            raise ValueError(f"--dump-outputs: {name} does not fit the {DUMP_BYTES} byte budget even as one row per frame")
        np.save(os.path.join(dirname, f"{name}.npy"), a)


def output_dumper(args, rank):
    """The --dump-outputs hook handed to a workload: rank 0 writes its own outputs; None without the flag and on other ranks."""
    if not args.dump_outputs or rank != 0:
        return None
    return lambda arrays: dump_outputs(args.dump_outputs, arrays)


def event_time_ms(torch, fn, iters):
    """Per-iteration CUDA-event durations (ms) of fn on the current stream, after two untimed calls (allocator, caches)."""
    fn()
    fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for s, e in evs:
        s.record()
        fn()
        e.record()
    torch.cuda.synchronize()
    return [s.elapsed_time(e) for s, e in evs]


def dist_setup(torch, n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        if os.environ.get("UPR_NO_NUMA_BIND", "") == "":
            from retinex_image_enhancement_b200 import native
            native.bind_to_gpu_numa_node(local)     # host buffers of the e2e legs land on the GPU's own NUMA node
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        return dist, rank, world, local
    if n_gpus > 1:
        raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one process per GPU)")
    torch.cuda.set_device(0)
    return None, 0, 1, 0


def barrier(torch, dist):
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(torch, dist, value: float) -> float:
    if dist is None:
        return value
    t = torch.tensor([value], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def timed_steps(torch, dist, fn, steps, warmup):
    """W untimed steps, then exactly K steps between barrier+sync on both sides; device time, max over ranks."""
    for _ in range(warmup):
        fn()
    barrier(torch, dist)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        fn()
    e.record()
    barrier(torch, dist)
    return max_over_ranks(torch, dist, s.elapsed_time(e))


def wall_steps(torch, dist, fn, steps, warmup):
    """Same bracket for host-synchronous calls (the host-buffer API returns when the result is on the host)."""
    for _ in range(warmup):
        fn()
    barrier(torch, dist)
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) * 1e3
    barrier(torch, dist)
    return max_over_ranks(torch, dist, dt)


# ---------------------------------------------------------------------------------------------------
# CPU arm: the reference's own path on the host cores
# ---------------------------------------------------------------------------------------------------
def cpu_frames(n, h, w, seed=1000):
    import numpy as np
    rng = np.random.default_rng(seed)
    x = rng.random((n, 3, h, w), dtype=np.float32)
    x[0::2] *= np.float32(0.3)
    return x


def find_reference():
    """Root of the unmodified reference tree, if one is at hand (never /root/reference on the GPU box: build() copies the tree
    to the git-ignored baseline/_ref, which travels with the repo snapshot)."""
    for root in (os.environ.get("UPR_REFERENCE"), os.path.join(ROOT, "baseline", "_ref"), "/root/reference"):
        if root and os.path.isfile(os.path.join(root, "enhancers", "adaptive_params.py")):
            return root
    return None


def load_reference_adjuster(root):
    """The reference's AdaptiveParameterAdjuster, imported from its own file, unmodified."""
    spec = importlib.util.spec_from_file_location("upr_reference_adaptive_params", os.path.join(root, "enhancers", "adaptive_params.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.AdaptiveParameterAdjuster()


def port_step_fn(workers):
    """The restated call sequence (oracle/cv2_chain.py) over a list of frames, `workers` frames at a time on a thread pool."""
    from oracle import cv2_chain
    cores = os.cpu_count() or 1
    if cv2_chain.available():
        import cv2
        cv2.setNumThreads(max(1, cores // max(workers, 1)))
        return (lambda xs: cv2_chain.clahe_lab_batch(xs, workers=workers)), f"oracle/cv2_chain.py (reference call sequence on cv2 {cv2.__version__} + numpy)"
    from oracle import oracle as O           # the cv2 wheel is absent: C restatement with OpenMP
    return (lambda xs: [O.clahe_lab(x) for x in xs]), "oracle/upr_oracle.c (C restatement, OpenMP)"


def cpu_reference_rate(h, w, budget_s=15.0, frames=None):
    """cpu_baseline of the b200 arm: Mpix/s of the reference CPU path on a bounded sample of the workload's frames.  The
    unmodified reference class (serial per-frame loop, OpenCV's own threading) when its tree is present, and the restated
    call sequence spread over every host core beside it."""
    import numpy as np
    cores = os.cpu_count() or 1
    workers = max(1, min(cores, 32))
    n = frames or max(workers, 8)
    xs = cpu_frames(n, h, w)
    out = {"unit": UNIT, "cores": cores}
    run_port, impl = port_step_fn(workers)
    run_port(xs[: max(1, min(n, workers))])  # warm-up (table init, thread pools)
    best, reps, t_start = None, 0, time.perf_counter()
    while reps < 5 and (time.perf_counter() - t_start) < budget_s * 0.5:
        t0 = time.perf_counter()
        run_port(xs)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
        reps += 1
    port = {"value": n * h * w / 1e6 / best, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n} frames {w}x{h} f32 of the same synthetic family, best of {reps} passes, {workers} worker threads; {impl}"}
    root = find_reference()
    if root is None:
        out.update(port)
        return out
    try:
        import cv2
        import torch
        cv2.setNumThreads(-1)                   # the reference's default: OpenCV threads across all cores
        adj = load_reference_adjuster(root)
        k = max(4, min(n, 8))
        ts = [torch.from_numpy(np.ascontiguousarray(x[None])) for x in xs[:k]]
        adj.apply_clahe_enhancement(ts[0])
        best_r, reps_r, t_start = None, 0, time.perf_counter()
        while reps_r < 3 and (time.perf_counter() - t_start) < budget_s * 0.5:
            t0 = time.perf_counter()
            for t in ts:
                adj.apply_clahe_enhancement(t)
            dt = time.perf_counter() - t0
            best_r = dt if best_r is None else min(best_r, dt)
            reps_r += 1
        out.update({"value": k * h * w / 1e6 / best_r, "kind": "reference",
                    "sample": f"{k} frames {w}x{h} f32, the unmodified AdaptiveParameterAdjuster.apply_clahe_enhancement from {root} in the "
                              f"reference's own serial per-frame loop (cv2 default threading), best of {reps_r} passes",
                    "port_threaded": port})
    except Exception as e:  # pragma: no cover
        out.update(port)
        out["reference_error"] = repr(e)
    return out


def run_reference_arm(args):
    """`--impl reference`: the reference's CPU implementation of the c2 step (64 x 1080p f32 frames through
    apply_clahe_enhancement, one by one) on the box's host cores; rank 0 only."""
    import numpy as np
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    h, w, n = C2_H, C2_W, C2_FRAMES
    cores = os.cpu_count() or 1
    xs = cpu_frames(n, h, w)
    root = find_reference()
    workers = max(1, min(cores, 32))
    run_port, impl = port_step_fn(workers)
    run_port(xs[:workers])
    t0 = time.perf_counter()
    run_port(xs)
    port_dt = time.perf_counter() - t0
    port = {"value": n * h * w / 1e6 / port_dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"one pass over the {n} frames, {workers} worker threads; {impl}"}
    kind, sample, step = "port", port["sample"], (lambda: run_port(xs))
    if root is not None:
        try:
            import cv2
            import torch
            cv2.setNumThreads(-1)
            adj = load_reference_adjuster(root)
            ts = [torch.from_numpy(np.ascontiguousarray(x[None])) for x in xs]

            def step():
                for t in ts:                          # enhancers/simple_enhance.py:237-243: one image after the other
                    adj.apply_clahe_enhancement(t)
            kind = "reference"
            sample = (f"{n} frames {w}x{h} f32 per step through the unmodified AdaptiveParameterAdjuster.apply_clahe_enhancement of {root}, "
                      f"the reference's own serial per-frame loop, cv2 {cv2.__version__} default threading on {cores} cores")
        except Exception as e:  # pragma: no cover
            sample += f" (reference import failed: {e!r})"
    warmup, steps = args.warmup, args.steps
    for _ in range(max(1, warmup)):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    mpix = steps * n * h * w / 1e6 / dt
    line = {"impl": "reference", "metric": METRIC, "value": mpix, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": dt * 1e3 / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8 fixed-point (f32 in/out)", "data": "synthetic", "config": dict(C2_CONFIG),
            "cpu_baseline": {"value": mpix, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "port_threaded": port},
            "e2e": {"value": mpix, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)
    return 0


# ---------------------------------------------------------------------------------------------------
# sub-records for the named BASELINE configs (also reachable as --workload c3|c4|c5)
# ---------------------------------------------------------------------------------------------------
class StubMaps:
    """CNN stand-in for the driver-level e2e leg (the CNN is out of scope): pointwise illumination / enhancement maps."""

    training = False

    def __init__(self, torch):
        self.torch = torch

    def forward_maps(self, x):
        return x.mean(dim=1, keepdim=True) * 0.5 + 0.25, self.torch.sqrt(x)


def record_c3(torch, dist, rank, world, local, steps, warmup, total_frames=256, dump=None):
    """BASELINE config 3: multi-scale statistics (a4) + gain/clamp (a5) on 256 4K frames sharded over the GPUs of the run
    (strong scaling: 256 / N frames per GPU; x read once, enhanced read, out written = 36 B/px)."""
    from retinex_image_enhancement_b200 import native
    h, w = 2160, 3840
    n = max(1, total_frames // world)
    dev = torch.device("cuda", local)
    x = make_frames(torch, n, h, w, 2000 + rank, dev)
    enh = torch.rand((n, 3, h, w), device=dev, generator=torch.Generator(device=dev).manual_seed(3000 + rank))
    out = torch.empty_like(enh)
    px = n * h * w
    last = []

    def step():
        last[:] = native.multiscale_enhance(x, enh, out=out)

    with ClockSampler(local) as clk:
        ms_step = timed_steps(torch, dist, step, steps, warmup) / steps
    if dump is not None:
        dump(dict(zip(("out", "means", "gain"), last)))
    k_stats = statistics.mean(event_time_ms(torch, lambda: native.multiscale_stats(x), 3))
    gain = native.multiscale_stats(x)[1]
    k_clamp = statistics.mean(event_time_ms(torch, lambda: native.scale_clamp(enh, gain, out=out), 3))
    peak, peak_src = measured_peak()
    dom = ("k_ms_stream", k_stats, 12.0) if k_stats >= k_clamp else ("k_gain_clamp_vec", k_clamp, 24.0)
    achieved = dom[2] * px / (dom[1] / 1e3) / 1e9
    rec = {"metric": "Mpix/s, 4K multi-scale statistics + gain (enhancers/multi_scale.py)", "value": world * px / 1e6 / (ms_step / 1e3),
           "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_step,
           "higher_is_better": True, "scaling": "strong", "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"c3: upr_multiscale_enhance_f32 (statistics kernel + gain/clamp kernel per ~25 Mpx chunk, two side streams) on "
                                  f"{total_frames} 3840x2160 f32 frames sharded by frame over {world} GPU(s) (CNN stubbed by a random 'enhanced' tensor)", "frames_per_gpu": n, "frames_total": n * world,
                      "h": h, "w": w, "l2": "inputs larger than L2"},
           "clocks": clk.summary(), "gpu_launches": 2 * -(-n // max(1, 25000000 // (h * w))) * steps,
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                        "kernel": dom[0], "kernel_ms": dom[1], "peak_source": peak_src,
                        "kernels_ms": {"k_ms_stream": k_stats, "k_gain_clamp_vec": k_clamp},
                        "op": {"algorithmic_bytes_per_px": 36, "achieved": 36.0 * px / (ms_step / 1e3) / 1e9,
                               "frac": 36.0 * px / (ms_step / 1e3) / 1e9 / peak}}}
    del x, enh, out
    torch.cuda.empty_cache()
    return rec


def record_c4(torch, dist, rank, world, local, steps, warmup, frames=8, size=256, extras=True, dump=None):
    """BASELINE config 4: texture statistics (a9/a10), per rank 8x3x256x256; the batch mean is one all-reduce of 2 floats.
    Latency bound: us/step for (kernel + NCCL all-reduce + weight kernel), the same as one CUDA graph, and for the ONE fused
    kernel that exchanges the pair over NVLink peer memory; and whether the three agree bit for bit."""
    from retinex_image_enhancement_b200 import native
    from retinex_image_enhancement_b200.losses import loss as L
    b, c, h, w = frames, 3, size, size
    dev = torch.device("cuda", local)
    x = torch.rand((b, c, h, w), device=dev, generator=torch.Generator(device=dev).manual_seed(11 + rank))

    # the product's default path (losses/loss.py DynamicSmoothWeight): one process = ONE kernel (statistics + batch mean + weight);
    # data-parallel = statistics kernel + NCCL all-reduce of [sum, count] + weight kernel
    default_dsw = L.DynamicSmoothWeight(1.0, True, "tv")
    last = []

    def step():
        last[:] = [default_dsw(x)]
        return last[0]

    def three_ops():
        _per, stats = L.batch_texture_stats(x, "tv")
        L.all_reduce_batch_stats(stats)
        return L.weight_from_stats(stats, 1.0)

    with ClockSampler(local) as clk:
        ms_step = timed_steps(torch, dist, step, steps, warmup) / steps
    if dump is not None:
        dump({"weight": last[0]})
    w_nccl = three_ops().clone()
    assert torch.equal(step(), w_nccl), "the one-kernel path and the three-operation path disagree"
    three_us = statistics.median(event_time_ms(torch, three_ops, 20)) * 1e3 if world == 1 else None
    # the same three operations captured in one CUDA graph (collective included when world > 1)
    graph_us = None
    try:
        step()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            wgt = step()
        ms_g = timed_steps(torch, dist, g.replay, steps, warmup) / steps
        graph_us = ms_g * 1e3
        del wgt
    except Exception as e:  # pragma: no cover
        graph_us = f"graph capture failed: {e!r}"
    # one kernel per rank: statistics + [sum, count] exchange over NVLink peer memory + weight (no NCCL call)
    fused_us, fused_equal = None, None
    try:
        dsw = L.DynamicSmoothWeight(1.0, True, "tv", fused_collective=True)
        w_fused = dsw(x).clone()
        fused_us = timed_steps(torch, dist, lambda: dsw(x), steps, warmup) / steps * 1e3
        eq = torch.tensor([1.0 if torch.equal(w_fused, w_nccl) else 0.0, float(abs(float(w_fused) - float(w_nccl)) <= 1e-6)], device=dev)
        if dist is not None:
            dist.all_reduce(eq, op=dist.ReduceOp.MIN)
        fused_equal = {"bit_equal_to_nccl_path_on_every_rank": bool(eq[0] > 0.5), "within_1e-6_of_nccl_path": bool(eq[1] > 0.5),
                       "note": "beyond two ranks NCCL's own summation order may differ from the kernel's rank order by 1 ulp"}
    except Exception as e:  # pragma: no cover
        fused_us = f"fused path failed: {e!r}"
    k_tv = statistics.mean(event_time_ms(torch, lambda: native.texture_complexity(x, "tv"), 20))
    k_ed = statistics.mean(event_time_ms(torch, lambda: native.texture_complexity(x, "edge_density"), 20))
    px = b * h * w
    peak, peak_src = measured_peak()
    achieved = 12.0 * px / (k_tv / 1e3) / 1e9
    rec = {"metric": "us per step, texture statistics + dynamic smoothness weight (losses/loss.py:523-583,704-720)",
           "value": ms_step * 1e3, "unit": "us/step", "higher_is_better": False, "mpix_s": world * px / 1e6 / (ms_step / 1e3),
           "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_step,
           "us_per_step": ms_step * 1e3, "us_per_step_cuda_graph": graph_us, "us_per_step_fused_peer_kernel": fused_us,
           "us_per_step_three_separate_ops": three_us,
           "fused_peer_vs_nccl": fused_equal, "scaling": "weak", "dtype": "f32 (fp64 accumulators)", "data": "synthetic",
           "config": {"workload": (f"c4: DynamicSmoothWeight on {b}x{c}x{h}x{w}: ONE kernel (upr_texture_weight_peer_f32: TV statistics + batch mean + weight)"
                                   if world == 1 else
                                   f"c4: upr_texture_tv_f32 on {b}x{c}x{h}x{w} per rank + all-reduce(SUM) of [sum, count] over {world} rank(s) + weight kernel"),
                      "l2": "latency-bound config (6.3 MB input is L2 resident by construction); reported in us/step"},
           "clocks": clk.summary(), "gpu_launches": (1 if world == 1 else 2) * steps,
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                        "kernel": "k_texture_tv", "kernel_ms": k_tv, "peak_source": peak_src,
                        "kernels_ms": {"k_texture_tv": k_tv, "k_texture_edge(1+2)": k_ed},
                        "note": "latency-bound at this size; see us_per_step"}}
    if extras:
        rec["smooth_loss"] = c4_loss_extras(torch, native, L, x, rank, dev)
    return rec


def c4_loss_extras(torch, native, L, x, rank, dev):
    """SURVEY 8f N3: the smoothness term and the statistics losses of the enhanced image beside the reference's torch ops."""
    b, _c, h, w = x.shape
    try:
        import torch.nn.functional as F
        illu = torch.rand((b, 1, h, w), device=dev, generator=torch.Generator(device=dev).manual_seed(21 + rank))
        mod = L.EdgeAwareSmoothnessLoss()
        ours = statistics.median(event_time_ms(torch, lambda: native.edge_smooth_loss(illu, x), 20)) * 1e3

        def stock():
            a = illu.detach().requires_grad_(True)
            mod._stock(a, x).backward()

        theirs = statistics.median(event_time_ms(torch, stock, 20)) * 1e3
        smooth = {"us_per_step": ours, "us_per_step_torch_ops_same_gpu": theirs, "api": "upr_edge_smooth_loss_f32 (loss + d loss / d illu)"}
        enh = torch.rand((b, 3, h, w), device=dev, generator=torch.Generator(device=dev).manual_seed(31 + rank))
        fused = L.EnhancedImageLosses()
        t_exp, t_col, t_spa = fused.exposure(), fused.color(), fused.spatial()

        def ours3():
            a = enh.detach().requires_grad_(True)
            (10.0 * t_exp(a, x) + 5.0 * t_col(a) + 1.0 * t_spa(a, x)).backward()

        def stock3():
            a = enh.detach().requires_grad_(True)
            gm = torch.mean(torch.mean(x, dim=1, keepdim=True))
            l_exp = torch.mean(torch.abs(F.avg_pool2d(torch.mean(a, dim=1, keepdim=True), 16, 16) - (0.6 + 0.2 * (1 - gm))))
            mr, mg, mb = (torch.mean(a[:, k]) for k in range(3))
            l_col = (mr - mg) ** 2 + (mr - mb) ** 2 + (mg - mb) ** 2
            dh = (a[..., :-1] - a[..., 1:]) - (x[..., :-1] - x[..., 1:])
            dv = (a[..., :-1, :] - a[..., 1:, :]) - (x[..., :-1, :] - x[..., 1:, :])
            (10.0 * l_exp + 5.0 * l_col + 1.0 * (torch.mean(dh ** 2) + torch.mean(dv ** 2))).backward()

        smooth["enhanced_image_losses"] = {"us_per_step": statistics.median(event_time_ms(torch, ours3, 20)) * 1e3,
                                           "us_per_step_torch_ops_same_gpu": statistics.median(event_time_ms(torch, stock3, 20)) * 1e3,
                                           "api": "upr_enh_losses_f32 + upr_enh_losses_grad_f32 through torch.autograd (exposure + colour + spatial)"}
        return smooth
    except Exception as e:  # pragma: no cover
        return {"error": repr(e)}


def record_c5(torch, dist, rank, world, local, steps, warmup, frames=128, chunk=16, dump=None):
    """BASELINE config 5: a stream of 4K frames, 128 per GPU (1024 over 8 GPUs), processed in chunks of 16 through the
    content-aware AND multi-scale enhancers chained in ONE call with ONE shared epilogue (upr_content_multiscale_f32: the
    multi-scale statistics run inside the chunk schedule of the content-aware passes):
    36 algorithmic B/px (x 12 + enhanced 12 read, out 12 written).  One step = the whole per-GPU stream."""
    from retinex_image_enhancement_b200 import native
    h, w = 2160, 3840
    n = frames
    dev = torch.device("cuda", local)
    x = make_frames(torch, n, h, w, 4000 + rank, dev)
    enh = torch.rand((n, 3, h, w), device=dev, generator=torch.Generator(device=dev).manual_seed(5000 + rank))
    out = torch.empty_like(enh)
    px = n * h * w
    chunks = [(a, min(a + chunk, n)) for a in range(0, n, chunk)]
    gains = [None] * len(chunks)

    def step():
        for i, (a, b) in enumerate(chunks):
            gains[i] = native.content_multiscale_apply(x[a:b], enh[a:b], out=out[a:b])[1]

    with ClockSampler(local) as clk:
        ms_step = timed_steps(torch, dist, step, steps, warmup) / steps
    if dump is not None:
        dump({"out": out, "gain": torch.cat(gains)})
    a, b = chunks[0]
    cpx = (b - a) * h * w
    k_ca = statistics.mean(event_time_ms(torch, lambda: native.content_aware_apply(x[a:b], enh[a:b], out=out[a:b]), 3))
    k_ms = statistics.mean(event_time_ms(torch, lambda: native.multiscale_stats(x[a:b]), 3))
    k_sal = statistics.mean(event_time_ms(torch, lambda: native.saliency(x[a:b]), 3))
    peak, peak_src = measured_peak()
    achieved = 36.0 * cpx / (k_ca / 1e3) / 1e9
    rec = {"metric": "Mpix/s, 4K content-aware + multi-scale enhance stream (enhancers/content_aware.py + multi_scale.py)",
           "value": world * px / 1e6 / (ms_step / 1e3), "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_step,
           "ms_per_chunk": ms_step / len(chunks), "higher_is_better": True, "scaling": "weak", "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"c5: {n} 3840x2160 f32 frames per GPU ({n * world} over {world} GPU(s)) in chunks of {chunk}: "
                                  "multi-scale statistics -> saliency blur -> raw attention -> ONE epilogue clamp(clamp(enh*(1+0.2 att))*gain), "
                                  "one call per chunk (upr_content_multiscale_f32)", "frames_per_gpu": n, "chunk": chunk, "h": h, "w": w,
                      "l2": "inputs larger than L2"},
           # per call: the library schedules sub-chunks of ~25 Mpx, each = statistics + min/max reset + blur + raw attention + epilogue kernels
           "clocks": clk.summary(), "gpu_launches": 5 * sum(-(-(b - a) // max(1, 25000000 // (h * w))) for a, b in chunks) * steps,
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                        "kernel": "upr_content_aware_apply_f32 chain (k_saliency_stream + k_sal_normalize + k_att_gain) on one chunk",
                        "kernel_ms": k_ca, "peak_source": peak_src, "algorithmic_bytes_per_px": 36,
                        "kernels_ms": {"content_aware_apply (3 passes)": k_ca, "k_ms_stream": k_ms, "saliency (blur + normalise)": k_sal},
                        "structural_note": "two global per-frame min/max dependencies force three passes that move 64 B/px: at most 0.56 of "
                                           "the 36 B/px roofline (profiles/r4_content_aware_l2.md)",
                        "op": {"algorithmic_bytes_per_px": 36, "achieved": 36.0 * px / (ms_step / 1e3) / 1e9,
                               "frac": 36.0 * px / (ms_step / 1e3) / 1e9 / peak,
                               "what": "content-aware + multi-scale chained, whole stream"}}}
    del x, enh, out
    torch.cuda.empty_cache()
    return rec


# ---------------------------------------------------------------------------------------------------
# the headline workload
# ---------------------------------------------------------------------------------------------------
def bench_c2(torch, dist, rank, world, local, args):
    from retinex_image_enhancement_b200 import native
    from retinex_image_enhancement_b200.enhancers.adaptive_params import AdaptiveParameterAdjuster
    from retinex_image_enhancement_b200.enhancers.simple_enhance import enhance_frames_host_u8

    n, h, w = args.frames or C2_FRAMES, C2_H, C2_W
    dev = torch.device("cuda", local)
    x = make_frames(torch, n, h, w, 1000 + rank, dev)
    out = torch.empty_like(x)
    px = n * h * w
    step = lambda: native.clahe_lab(x, out=out)  # noqa: E731

    with ClockSampler(local) as clk:
        ms_total = timed_steps(torch, dist, step, args.steps, args.warmup)
    dump = output_dumper(args, rank)
    if dump is not None:
        dump({"out": out})      # before the kernel legs below overwrite `out`
    ms_step = ms_total / args.steps
    value = world * px / 1e6 / (ms_step / 1e3)

    # per-kernel durations, live, CUDA events on the launching stream (profiling hook of the C ABI)
    with ClockSampler(local) as clk_legs:
        k1 = statistics.mean(event_time_ms(torch, lambda: native.clahe_lab(x, out=out, stage_mask=1), max(5, args.steps // 2)))
        k3 = statistics.mean(event_time_ms(torch, lambda: native.clahe_lab(x, out=out, stage_mask=2), max(5, args.steps // 2)))
    peak, peak_src = measured_peak()
    # algorithmic bytes of each kernel: K1 reads the f32 frame (12 B/px); K3 writes the f32 frame (12 B/px);
    # the 3 B/px u8 Lab intermediate between them is NOT algorithmic (it is what `traffic` exposes)
    dom_name, dom_ms = ("k_map_vec5", k3) if k3 >= k1 else ("k_hist_lab_vec3", k1)
    alg_bytes = 12.0 * px
    achieved = alg_bytes / (dom_ms / 1e3) / 1e9
    op_achieved = 24.0 * px / (ms_step / 1e3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": args.traffic if args.traffic is not None else committed_traffic(dom_name), "kernel": dom_name, "kernel_ms": dom_ms, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes,
                "kernels_ms": {"k_hist_lab_vec3": k1, "k_map_vec5": k3}, "kernel_legs_clocks": clk_legs.summary(),
                "op": {"algorithmic_bytes_per_px": 24, "achieved": op_achieved, "frac": op_achieved / peak,
                       "frac_of_nominal_8000": op_achieved / 8000.0}}

    # the Retinex arithmetic of the same configuration (a8, models/model.py:405-413,442), reported separately (SURVEY 8d):
    # R = x / (illu + 1e-6), enh = R*e + (1-R)*e^2 without materialising R: 12 + 4 + 12 read, 12 written = 40 B/px
    illu = (x[:, :1] * 0.5 + 0.25).contiguous()
    k8 = statistics.median(event_time_ms(torch, lambda: native.retinex_recombine(x, illu, out, want_reflectance=False), 9))
    roofline["retinex_recombine"] = {"kernel": "k_recombine_vec", "kernel_ms": k8, "algorithmic_bytes_per_px": 40,
                                     "achieved": 40.0 * px / (k8 / 1e3) / 1e9, "frac": 40.0 * px / (k8 / 1e3) / 1e9 / peak}
    # the enhance path after the CNN in ONE call (upr_retinex_clahe_f32): recombination in the registers of the histogram
    # kernel + CLAHE; 40 B/px (x 12 + illu 4 + e 12 read, out 12 written) instead of 64 B/px for the two ops back to back
    e_map = torch.rand((n, 3, h, w), device=dev, generator=torch.Generator(device=dev).manual_seed(7000 + rank))
    kf = statistics.median(event_time_ms(torch, lambda: native.retinex_clahe(x, illu, e_map, out=out), 9))
    roofline["fused_enhance"] = {"api": "upr_retinex_clahe_f32 (k_hist_lab_vec3<fused Retinex prologue> + k_map_vec5)", "ms": kf,
                                 "mpix_s": px / 1e6 / (kf / 1e3), "algorithmic_bytes_per_px": 40,
                                 "achieved": 40.0 * px / (kf / 1e3) / 1e9, "frac": 40.0 * px / (kf / 1e3) / 1e9 / peak,
                                 "unfused_ms": k8 + ms_step}
    del illu, e_map

    # end to end through the reference-facing API with host tensors
    adj = AdaptiveParameterAdjuster()
    n_e2e = n
    hx = torch.empty((n_e2e, 3, h, w), dtype=torch.float32, pin_memory=True)
    hx.copy_(x[:n_e2e])
    e2e_steps = max(2, min(args.steps, 20))     # exactly K steps up to 20 (a step is 36 ms of PCIe traffic at the f32 boundary)
    ms_e2e = wall_steps(torch, dist, lambda: adj.apply_clahe_enhancement(hx), e2e_steps, max(2, min(args.warmup, 3))) / e2e_steps
    e2e = {"value": world * n_e2e * h * w / 1e6 / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": hx.numel() * 4,
           "d2h_bytes_per_step": hx.numel() * 4, "ms_per_step": ms_e2e, "steps": e2e_steps,
           "api": "AdaptiveParameterAdjuster.apply_clahe_enhancement(host f32 [64,3,1080,1920]) -> host tensor "
                  "(upr_clahe_lab_f32_host, pinned buffers, 3-stream chunk pipeline)",
           "note": "PCIe-bound: 12 + 12 B/px cross the host link; on this pool's virtualised hosts the link saturates near 68 GB/s per "
                   "direction for the whole box, so this figure does not scale with the GPU count (see e2e_driver for the 3 + 4 B/px boundary)"}
    del hx

    # the same op at the packed u8 boundary (upr_clahe_lab_u8: what image files decode to / are saved as; 3 + 3 B/px instead of
    # 12 + 12 over PCIe).  Reported beside the headline, which stays on the reference's f32 tensor API.
    x8 = (x * 255.0).to(torch.uint8).permute(0, 2, 3, 1).contiguous()
    o8 = torch.empty_like(x8)
    ku8 = statistics.median(event_time_ms(torch, lambda: native.clahe_lab_u8(x8, out=o8), 9))
    hx8 = torch.empty(x8.shape, dtype=torch.uint8, pin_memory=True)
    hx8.copy_(x8)
    ho8 = torch.empty(x8.shape, dtype=torch.uint8, pin_memory=True)
    ms_e2e8 = wall_steps(torch, dist, lambda: native.clahe_lab_u8_host(hx8, out=ho8), e2e_steps, max(2, min(args.warmup, 3))) / e2e_steps
    u8_boundary = {"api": "upr_clahe_lab_u8 / upr_clahe_lab_u8_host (packed u8 RGB, HWC)", "device_ms": ku8,
                   "device_mpix_s": world * px / 1e6 / (ku8 / 1e3),
                   "e2e": {"value": world * px / 1e6 / (ms_e2e8 / 1e3), "unit": UNIT, "ms_per_step": ms_e2e8,
                           "h2d_bytes_per_step": hx8.numel(), "d2h_bytes_per_step": hx8.numel()}}
    del x8, o8

    # the enhance DRIVER end to end (enhancers/simple_enhance.py, SURVEY 8f N1): host uint8 frames as decoded -> upload ->
    # de-quantise -> (CNN stubbed) -> Retinex recombination + CLAHE fused, u8 out of the map kernel -> illumination u8 ->
    # download: what enhance_batch_images does between its decode and PNG thread pools
    ho_illu = torch.empty((n, h, w, 1), dtype=torch.uint8, pin_memory=True)
    stub = StubMaps(torch)

    def driver_step():
        for ev in enhance_frames_host_u8(stub, hx8, ho8, ho_illu, dev, chunk=8):
            ev.synchronize()

    ms_drv = wall_steps(torch, dist, driver_step, e2e_steps, max(2, min(args.warmup, 3))) / e2e_steps
    e2e_driver = {"value": world * px / 1e6 / (ms_drv / 1e3), "unit": UNIT, "ms_per_step": ms_drv, "steps": e2e_steps,
                  "h2d_bytes_per_step": hx8.numel(), "d2h_bytes_per_step": ho8.numel() + ho_illu.numel(),
                  "api": "enhancers.simple_enhance.enhance_frames_host_u8(host u8 [64,1080,1920,3]) -> host u8 enhanced + illumination "
                         "(upr_letterbox_u8_f32 -> stub CNN maps -> upr_retinex_clahe_f32_u8 -> upr_quantize_u8_f32; chunks of 8 over 3 streams)",
                  "note": "CNN stubbed by pointwise maps (out of scope); 3 B/px up, 4 B/px down"}
    if rank == 0 and not args.no_cpu:
        # the CPU chain at the same boundary: the OpenCV calls alone on u8 frames (no float casts), every host core
        try:
            from oracle import cv2_chain
            if cv2_chain.available():
                import cv2
                cores = os.cpu_count() or 1
                workers = max(1, min(cores, 32))
                cv2.setNumThreads(max(1, cores // workers))
                sample = hx8[: max(workers, 8)].numpy()
                cv2_chain.clahe_lab_batch_u8(sample[:workers], workers=workers)
                best = None
                for _ in range(3):
                    t0 = time.perf_counter()
                    cv2_chain.clahe_lab_batch_u8(sample, workers=workers)
                    dt = time.perf_counter() - t0
                    best = dt if best is None else min(best, dt)
                u8_boundary["cpu_baseline"] = {"value": sample.shape[0] * h * w / 1e6 / best, "unit": UNIT, "cores": cores, "kind": "port",
                                               "sample": f"{sample.shape[0]} u8 frames, best of 3, {workers} worker threads; "
                                                         "oracle/cv2_chain.py clahe_lab_batch_u8 (the reference's OpenCV calls alone)"}
        except Exception as e:  # pragma: no cover
            u8_boundary["cpu_baseline"] = {"error": repr(e)}
    del hx8, ho8, ho_illu

    cpu = cpu_reference_rate(h, w, budget_s=args.cpu_budget) if rank == 0 and not args.no_cpu else None
    del x, out
    torch.cuda.empty_cache()

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8 fixed-point (f32 in/out)", "data": "synthetic", "config": dict(C2_CONFIG),
            "clocks": clk.summary(), "e2e": e2e, "e2e_driver": e2e_driver, "gpu_launches": 2 * args.steps, "roofline": roofline,
            "u8_boundary": u8_boundary}
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if not args.no_named:
        # the other BASELINE configs at this run's GPU count (every rank takes part; rank 0 reports)
        named = {}
        sub_steps = max(3, min(args.steps, 10))
        for name, fn in (("c3", lambda: record_c3(torch, dist, rank, world, local, sub_steps, 3)),
                         ("c4", lambda: record_c4(torch, dist, rank, world, local, max(args.steps, 50), 5, extras=False)),
                         ("c5", lambda: record_c5(torch, dist, rank, world, local, max(3, sub_steps // 2), 3))):
            try:
                named[name] = fn()
            except Exception as e:  # pragma: no cover
                named[name] = {"error": repr(e)}
                torch.cuda.empty_cache()
        line["named_configs"] = named
    return line


def bench_c3(torch, dist, rank, world, local, args):
    rec = record_c3(torch, dist, rank, world, local, args.steps, args.warmup, total_frames=(args.frames * world) if args.frames else 256,
                    dump=output_dumper(args, rank))
    rec["vs_baseline"] = None
    return rec


def bench_c4(torch, dist, rank, world, local, args):
    rec = record_c4(torch, dist, rank, world, local, args.steps, args.warmup, frames=args.frames or 8, size=args.size or 256,
                    dump=output_dumper(args, rank))
    rec["vs_baseline"] = None
    return rec


def bench_c5(torch, dist, rank, world, local, args):
    rec = record_c5(torch, dist, rank, world, local, args.steps, args.warmup, frames=args.frames or 128, dump=output_dumper(args, rank))
    rec["vs_baseline"] = None
    return rec


WORKLOADS = {"c2": bench_c2, "c3": bench_c3, "c4": bench_c4, "c5": bench_c5}


_RESULT_OUT = None


def claim_stdout():
    """stdout must carry exactly ONE JSON line.  Libraries write there too (NCCL prints its version banner on stdout at
    NCCL_DEBUG=VERSION/WARN), so file descriptor 1 is pointed at stderr for the whole run and the result line goes to a
    duplicate of the original stdout."""
    global _RESULT_OUT
    if _RESULT_OUT is None:
        sys.stdout.flush()
        _RESULT_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    return _RESULT_OUT


def emit(line):
    out = claim_stdout()
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--frames", type=int, default=0, help="frames per GPU (default: the workload's own)")
    ap.add_argument("--size", type=int, default=0, help="c4 only: image side")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-named", action="store_true", help="c2 only: skip the named_configs sub-records (c3, c4, c5)")
    ap.add_argument("--cpu-budget", type=float, default=15.0)
    ap.add_argument("--traffic", type=float, default=None,
                    help="dram bytes per launch of the dominant kernel from the committed ncu capture (profiles/)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy (rank 0; a fixed sample of "
                         "outputs over 1 MB, at most 48 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: upretinex-b200 has no CPU path (use --impl reference for the CPU arm)")
    import __graft_entry__ as entry
    entry.ensure_built()
    dist, rank, world, local = dist_setup(torch, args.gpus)
    try:
        line = WORKLOADS[args.workload](torch, dist, rank, world, local, args)
        if rank == 0:
            emit(line)
    finally:
        if dist is not None:
            dist.destroy_process_group()
    return 0


def committed_traffic(kernel=None):
    """dram bytes per launch of a kernel (default: the dominant one), read from the committed ncu summary (profiles/), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            d = json.load(f)
        if kernel is not None and kernel in d.get("kernels", {}):
            return float(d["kernels"][kernel])
        return float(d["dominant_kernel_dram_bytes_per_launch"])
    except Exception:
        return None


if __name__ == "__main__":
    sys.exit(main())
