"""Drop-in for the reference's ``enhancers/simple_enhance.py`` drivers (same function names, argument order,
defaults and output file names ``{stem}_enhanced.png``, ``{stem}_illumination.png``, ``{stem}_comparison.png``).

Reference (file:line relative to the reference tree): load_image :23-62, save_image :65-100, create_comparison
:103-132, enhance_single_image :135-199, enhance_batch_images :202-250.

B200-first differences:
  * frames cross PCIe as uint8 in BOTH directions: the decoded file goes up as it is (3 B/px) and is de-quantised /
    letterboxed on the device (upr_letterbox_u8_f32); what comes back is the frame ``save_image`` would store, quantised
    on the device -- by the CLAHE map kernel itself on the default path (upr_retinex_clahe_f32_u8 / upr_clahe_lab_f32_u8),
    by upr_quantize_u8_f32 otherwise -- plus the 1 B/px illumination map.  The reference moves 12 B/px three times per
    image (adaptive_params.py:188/:136/:198);
  * ``enhance_batch_images`` is a three-stage pipeline (SURVEY 8f row N1): a thread pool decodes files ahead of the GPU into
    host arrays, same-shaped frames are packed into pinned double-buffered staging and run as ONE device batch on a side
    stream, and PNG encoding runs on a second thread pool that waits on the batch's CUDA event -- decode, GPU work and
    encode of neighbouring batches overlap.  It honours ``enable_multi_scale`` / ``enable_content_aware`` (the reference
    silently drops them at :240) and, launched with one process per GPU (torchrun), shards the file list by rank and binds
    each rank to cuda:LOCAL_RANK -- frames are independent, there is no collective;
  * ``enhance_single_image`` accepts ``adjuster=`` (the reference's main.py:246 passes it and crashes on the missing
    parameter);
  * ``amp="fp16"`` / ``"bf16"`` runs the CNN and the fused Retinex + CLAHE dispatch under ``torch.autocast("cuda")``; the
    fp16 / bf16 maps go straight into the fused kernels (default None: f32, the reference's behaviour).
File decoding / PNG encoding themselves stay PIL (an nvJPEG decode would not be bit-identical to the reference's).
"""
from __future__ import annotations

import contextlib
import os
import time
from collections import deque

import numpy as np
import torch

from ..models.model import UP_Retinex
from ..utils.letterbox import letterbox_geometry, letterbox_tensor
from .adaptive_params import AdaptiveParameterAdjuster, cnn_maps
from .content_aware import ContentAwareEnhancer
from .multi_scale import MultiScaleEnhancer

VALID_EXTENSIONS = {".jpg", ".jpeg", ".png", ".bmp", ".tif", ".tiff"}
AMP_DTYPES = {"fp16": torch.float16, "bf16": torch.bfloat16}


def amp_context(amp):
    """torch.autocast("cuda") in the dtype that ``amp`` names ("fp16" / "bf16"); no context for None."""
    if amp is None:
        return contextlib.nullcontext()
    if amp not in AMP_DTYPES:
        raise ValueError(f"amp must be None, 'fp16' or 'bf16', got {amp!r}")
    return torch.autocast("cuda", dtype=AMP_DTYPES[amp])


def bind_rank_to_gpu() -> str:
    """One process per GPU (torchrun): bind this process to cuda:LOCAL_RANK (and to the CPU cores next to that GPU, so that
    pinned staging buffers are first-touched on its NUMA node) and return the device string the drivers should use.  Without
    LOCAL_RANK / WORLD_SIZE in the environment it is the current device."""
    if not torch.cuda.is_available():
        return "cpu"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 or "LOCAL_RANK" in os.environ:
        local = int(os.environ.get("LOCAL_RANK", "0"))
        count = torch.cuda.device_count()
        if local >= count:
            raise RuntimeError(f"LOCAL_RANK={local} but only {count} CUDA device(s) are visible: launch one process per GPU")
        torch.cuda.set_device(local)
        from .. import native
        native.bind_to_gpu_numa_node(local)
        return f"cuda:{local}"
    return f"cuda:{torch.cuda.current_device()}"


def resolve_device(device) -> str:
    """'cuda' / None under torchrun -> this rank's own GPU; anything explicit ('cuda:3', 'cpu') is taken as given."""
    if device is None or str(device) == "cuda":
        return bind_rank_to_gpu() if torch.cuda.is_available() else (device or "cpu")
    return str(device)


def _decode_u8(image_path):
    """File -> contiguous uint8 [H,W,3] array and the file's (W, H), decoded like the reference (PIL, RGB)."""
    from PIL import Image
    img = Image.open(image_path).convert("RGB")
    return np.array(img, dtype=np.uint8), img.size      # (a writable copy: torch.from_numpy refuses read-only buffers)


def _geometry(h, w, max_size):
    """(resized hw, (top, left), output hw) of the reference's letterbox call (enhancers/simple_enhance.py:43-58)."""
    if max_size is None:
        return (h, w), (0, 0), (h, w)
    (rh, rw), (top, bottom, left, right), _, _ = letterbox_geometry(h, w, max_size, auto=True, scaleup=False)
    return (rh, rw), (top, left), (rh + top + bottom, rw + left + right)


def load_image(image_path, max_size=None, device=None):
    """-> ([1,3,H,W] f32 tensor in [0,1], (W, H) of the file).  Host tensor like the reference's by default.  With a CUDA
    ``device`` (what the drivers below pass) the decoded uint8 frame is uploaded as is -- 3 instead of 12 bytes per pixel
    over PCIe -- and de-quantised / letterboxed on the device (upr_letterbox_u8_f32; same values, bit for bit)."""
    arr, original_size = _decode_u8(image_path)
    if device is not None and torch.device(device).type == "cuda":
        from .. import native
        u8 = torch.from_numpy(arr).unsqueeze(0)
        (rh, rw), (top, left), out_hw = _geometry(u8.shape[1], u8.shape[2], max_size)
        dev = torch.device(device)
        with torch.cuda.device(dev):
            t = native.letterbox(u8.pin_memory().to(dev, non_blocking=True), (rh, rw), top, left, out_hw)
        return t, original_size
    t = torch.from_numpy(arr).permute(2, 0, 1).to(torch.float32) / 255.0
    if max_size is not None:
        t, _, _ = letterbox_tensor(t, new_shape=max_size, auto=True, scaleup=False)
    # max_size None: letterbox to the image's own shape is the identity on a k/255 grid (see utils/letterbox.py)
    return t.unsqueeze(0).contiguous(), original_size


def _to_u8_hwc(tensor):
    """[1,C,H,W] / [C,H,W] f32 -> [H,W,3] uint8 array: (clip(x,0,1)*255).astype(uint8) as in the reference's save_image
    (enhancers/simple_enhance.py:65-80).  A CUDA tensor is clipped, quantised and interleaved by upr_quantize_u8_f32, so only
    1 or 3 bytes per pixel cross PCIe (the same truncating cast; uint8 arrays pass through, single-channel ones tripled)."""
    if isinstance(tensor, np.ndarray):
        a = tensor
        if a.ndim == 3 and a.shape[2] == 1:
            a = np.repeat(a, 3, axis=2)
        return a
    if tensor.dim() == 4:
        tensor = tensor.squeeze(0)
    t = tensor.detach().to(torch.float32)
    if t.is_cuda:
        from .. import native
        with torch.cuda.device(t.device):
            q = native.quantize_u8(t.unsqueeze(0).contiguous())[0].cpu().numpy()
        return np.repeat(q, 3, axis=2) if q.shape[2] == 1 else q
    a = (np.clip(t.numpy(), 0, 1) * 255).astype(np.uint8)
    if a.shape[0] == 1:
        return np.stack([a[0]] * 3, axis=2)
    return np.transpose(a, (1, 2, 0))


def save_image(tensor, save_path):
    from PIL import Image
    Image.fromarray(_to_u8_hwc(tensor)).save(save_path)
    print(f"已保存: {save_path}")


def create_comparison(img_low, img_enhanced, save_path):
    from PIL import Image
    Image.fromarray(np.concatenate([_to_u8_hwc(img_low), _to_u8_hwc(img_enhanced)], axis=1)).save(save_path)
    print(f"已保存对比图像: {save_path}")


def _enhance_tensor(model, img_low, device, enable_multi_scale, enable_content_aware, adjuster=None):
    """Dispatch of enhancers/simple_enhance.py:167-175 on a [N,3,H,W] batch."""
    if enable_content_aware:
        return ContentAwareEnhancer().apply_content_aware_enhancement(model, img_low, device)
    if enable_multi_scale:
        return MultiScaleEnhancer().enhance_with_pyramid(model, img_low, device)
    return (adjuster or AdaptiveParameterAdjuster()).apply_adaptive_enhancement(model, img_low, device)


def enhance_frames_u8(model, low, enable_multi_scale=False, enable_content_aware=False, adjuster=None,
                      out_enh=None, out_illu=None):
    """The same dispatch with the STORED frames as the result: low [N,3,H,W] f32 CUDA -> (enhanced [N,H,W,3] u8,
    illumination [N,H,W,1] u8), both on the device, exactly the bytes ``save_image`` would write for the f32 results of
    ``_enhance_tensor``.  On the default (CLAHE) path the map kernel emits the u8 frame itself."""
    from .. import native
    with torch.no_grad():
        if not (enable_content_aware or enable_multi_scale):
            adj = adjuster or AdaptiveParameterAdjuster()
            adj.note_input(low)
            if hasattr(model, "forward_maps") and not getattr(model, "training", False):
                illu, e_map = model.forward_maps(low)
                enh8 = native.retinex_clahe_u8(low.contiguous(), illu.contiguous(), e_map.contiguous(), adj.CLIP_LIMIT, adj.TILE_GRID,
                                               out=out_enh, autocast=torch.is_autocast_enabled("cuda"))
            else:
                enhanced, _refl, illu = model(low)
                enh8 = native.clahe_lab_f32_u8(enhanced.contiguous(), adj.CLIP_LIMIT, adj.TILE_GRID, out=out_enh)
        else:
            maps = cnn_maps(model, low)
            if maps is not None:
                # both stored frames from the mode's last pass (content-aware wins when both flags are set, as in
                # _enhance_tensor); the illumination frame is the widened map quantised, as below
                fn = native.retinex_content_aware_u8 if enable_content_aware else native.retinex_multiscale_u8
                return fn(low.contiguous(), *maps, autocast=torch.is_autocast_enabled("cuda"), out=out_enh, out_illu=out_illu)
            enhanced, illu = _enhance_tensor(model, low, low.device, enable_multi_scale, enable_content_aware)
            enh8 = native.quantize_u8(enhanced.contiguous(), out=out_enh)
        # a map from a CNN under autocast is widened first, as _to_u8_hwc does
        illu8 = native.quantize_u8(illu.to(torch.float32).contiguous(), out=out_illu)
    return enh8, illu8


_stream_rings = {}


def _stream_ring(dev, count=3):
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), count)
    ring = _stream_rings.get(key)
    if ring is None:
        ring = [torch.cuda.Stream(device=dev) for _ in range(count)]
        _stream_rings[key] = ring
    return ring


def _chunk_bounds(n, chunk):
    """[(f0, f1)] covering n frames in chunks of ``chunk`` with a half-sized first and last chunk: the first upload and the last
    download of the pipeline overlap with nothing, so both ends are kept short."""
    chunk = max(1, int(chunk))
    edge = max(1, chunk // 2) if n > 2 * chunk else chunk
    bounds, f0, first = [], 0, True
    while f0 < n:
        left = n - f0
        nf = edge if first else chunk
        if left - nf < edge < left:
            nf = left - edge          # leave exactly ``edge`` frames for the last chunk
        nf = min(nf, left)
        bounds.append((f0, f0 + nf))
        f0 += nf
        first = False
    return bounds


def enhance_frames_host_u8(model, frames_u8, out_enh, out_illu, device, max_size=None, enable_multi_scale=False,
                           enable_content_aware=False, out_low=None, chunk=8, frame_fn=None):
    """The device side of the batch driver, end to end at the uint8 boundary: HOST frames as decoded ([N,H,W,3] u8, pinned for
    full PCIe speed) -> HOST frames as ``save_image`` would store them (``out_enh`` [N,H',W',3] u8, ``out_illu`` [N,H',W',1] u8;
    ``out_low`` [N,H',W',3] receives the letterboxed input when ``max_size`` changes it).  The batch is cut into chunks of
    ``chunk`` frames that rotate over three CUDA streams: the upload of chunk k+1 and the download of chunk k-1 overlap the
    kernels of chunk k; 3 B/px go up, 4 B/px come back.  Returns the CUDA events of the chunks, in order: ``event.synchronize()``
    before reading the corresponding frames of the output buffers (the PNG writers of enhance_batch_images do exactly that).
    ``frame_fn(low [n,3,H',W'] f32 CUDA) -> (enhanced u8 [n,H',W',3], illumination u8 [n,H',W',1])`` replaces the enhancer dispatch
    (predict_batch passes the bare model)."""
    from .. import native
    dev = torch.device(resolve_device(device))
    n, h, w = frames_u8.shape[0], frames_u8.shape[1], frames_u8.shape[2]
    (rh, rw), (top, left), out_hw = _geometry(h, w, max_size)
    ring = _stream_ring(dev)
    launch = torch.cuda.current_stream(dev)
    ready = torch.cuda.Event()
    ready.record(launch)
    events = []
    with torch.cuda.device(dev):
        for k, (f0, f1) in enumerate(_chunk_bounds(n, chunk)):
            st = ring[k % len(ring)]
            st.wait_event(ready)
            with torch.cuda.stream(st):
                low = native.letterbox(frames_u8[f0:f1].to(dev, non_blocking=True), (rh, rw), top, left, out_hw)
                enh8, illu8 = frame_fn(low) if frame_fn is not None else enhance_frames_u8(model, low, enable_multi_scale, enable_content_aware)
                out_enh[f0:f1].copy_(enh8, non_blocking=True)
                out_illu[f0:f1].copy_(illu8, non_blocking=True)
                if out_low is not None:
                    out_low[f0:f1].copy_(native.quantize_u8(low), non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(st)
            events.append(ev)
    return events


def _write_outputs(img_low, img_enhanced, illu_map, image_path, output_dir, pool=None):
    """The reference's three files per image (enhancers/simple_enhance.py:177-195).  Quantisation happens here (on the
    device for CUDA tensors); with ``pool`` (a ThreadPoolExecutor) the PNG encoding runs on host threads."""
    os.makedirs(output_dir, exist_ok=True)
    stem = os.path.splitext(os.path.basename(image_path))[0]
    low, enh, illu = _to_u8_hwc(img_low), _to_u8_hwc(img_enhanced), _to_u8_hwc(illu_map)

    def write():
        save_image(enh, os.path.join(output_dir, f"{stem}_enhanced.png"))
        save_image(illu, os.path.join(output_dir, f"{stem}_illumination.png"))
        create_comparison(low, enh, os.path.join(output_dir, f"{stem}_comparison.png"))

    if pool is None:
        write()
        return None
    return pool.submit(write)


def enhance_single_image(model, image_path, output_dir, device, max_size=None, enable_multi_scale=False,
                         enable_content_aware=False, adjuster=None, amp=None):
    print(f"正在处理: {os.path.basename(image_path)}")
    device = resolve_device(device)
    img_low, _original_size = load_image(image_path, max_size, device=device)
    start = time.time()
    with amp_context(amp):
        img_enhanced, illu_map = _enhance_tensor(model, img_low, device, enable_multi_scale, enable_content_aware, adjuster)
    if img_enhanced.is_cuda:
        torch.cuda.synchronize(img_enhanced.device)
    print(f"增强耗时: {time.time() - start:.4f}s")
    _write_outputs(img_low, img_enhanced, illu_map, image_path, output_dir)
    print("图像增强完成！")


def list_images(input_dir):
    return sorted(os.path.join(input_dir, f) for f in os.listdir(input_dir)
                  if os.path.splitext(f)[1].lower() in VALID_EXTENSIONS)


def shard_for_rank(items, rank=None, world=None):
    """Contiguous block of ``items`` owned by this rank (frame i -> GPU i*G/N; no collective on the enhance path)."""
    if rank is None or world is None:
        rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    n = len(items)
    lo, hi = (n * rank) // world, (n * (rank + 1)) // world
    return items[lo:hi]


class _Staging:
    """Two pinned (input u8, enhanced u8, illumination u8[, letterboxed input u8]) buffer sets per frame shape: while the
    writers still read set k, the GPU fills set k^1.  A set is reused only after the PNG tasks that read it have finished."""

    def __init__(self, batch_size):
        self.batch_size = batch_size
        self.sets = {}

    def acquire(self, in_hw, out_hw, want_low):
        key = (in_hw, out_hw, want_low)
        ring = self.sets.setdefault(key, {"next": 0, "slots": [None, None]})
        k = ring["next"]
        ring["next"] = k ^ 1
        slot = ring["slots"][k]
        if slot is None:
            b = self.batch_size
            pin = lambda *shape: torch.empty(shape, dtype=torch.uint8, pin_memory=True)  # noqa: E731
            slot = {"in": pin(b, in_hw[0], in_hw[1], 3), "enh": pin(b, out_hw[0], out_hw[1], 3), "illu": pin(b, out_hw[0], out_hw[1], 1),
                    "low": pin(b, out_hw[0], out_hw[1], 3) if want_low else None, "readers": []}
            ring["slots"][k] = slot
        for fut in slot["readers"]:
            fut.result()
        slot["readers"] = []
        return slot


def run_batch_pipeline(files, output_dir, device, max_size, batch_size, frame_fn, write_files, host_fn,
                       decode_workers=None, encode_workers=None):
    """The three-stage pipeline behind enhance_batch_images and predict_batch: decode pool -> pinned double-buffered u8 staging ->
    one device batch per run of same-shaped frames (``frame_fn``, see enhance_frames_host_u8) -> PNG pool (``write_files(stem,
    low8, enh8, illu8)`` runs on a writer thread once the batch's CUDA event has fired).  ``host_fn(path, u8 array)`` handles a
    frame when ``device`` is not a CUDA device."""
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(output_dir, exist_ok=True)
    on_gpu = torch.device(device).type == "cuda"
    cores = os.cpu_count() or 1
    decoders = ThreadPoolExecutor(max_workers=decode_workers or min(8, cores))
    writers = ThreadPoolExecutor(max_workers=encode_workers or min(8, cores))
    futures, last_write_of_stem = [], {}

    def submit_write(stem, task):
        """PNG tasks of inputs that share a stem (a.jpg and a.png) target the same files: chain them so that they are written
        one after the other, in list order, like the reference's sequential loop (the last one wins)."""
        prev = last_write_of_stem.get(stem)

        def run():
            if prev is not None:
                prev.result()
            task()
        fut = writers.submit(run)
        last_write_of_stem[stem] = fut
        futures.append(fut)
        return fut

    staging = _Staging(batch_size)

    def run_batch(batch):
        """batch: list of (path, u8 HWC array) of one shape."""
        if not on_gpu:
            for path, arr in batch:
                host_fn(path, arr)
            return
        b = len(batch)
        h, w = batch[0][1].shape[:2]
        (rh, rw), (top, left), out_hw = _geometry(h, w, max_size)
        identity = out_hw == (h, w) and (rh, rw) == (h, w)
        slot = staging.acquire((h, w), out_hw, not identity)
        for i, (_p, arr) in enumerate(batch):
            slot["in"][i].copy_(torch.from_numpy(arr))
        event = enhance_frames_host_u8(None, slot["in"][:b], slot["enh"][:b], slot["illu"][:b], device, max_size,
                                       out_low=None if identity else slot["low"][:b], chunk=b, frame_fn=frame_fn)[-1]
        for i, (path, arr) in enumerate(batch):
            stem = os.path.splitext(os.path.basename(path))[0]
            low8 = arr if identity else slot["low"][i].numpy()      # un-letterboxed: the decoded bytes ARE the stored input
            enh8, illu8 = slot["enh"][i].numpy(), slot["illu"][i].numpy()

            def task(stem=stem, low8=low8, enh8=enh8, illu8=illu8):
                event.synchronize()          # the batch's D2H copies have landed in the pinned buffers
                write_files(stem, low8, enh8, illu8)
            slot["readers"].append(submit_write(stem, task))

    try:
        window = deque()
        ahead = max(2 * batch_size, 4)
        it = iter(files)
        pending = []            # consecutive same-shape frames form one device batch

        def top_up():
            while len(window) < ahead:
                path = next(it, None)
                if path is None:
                    return
                window.append((path, decoders.submit(_decode_u8, path)))

        top_up()
        while window:
            path, fut = window.popleft()
            arr, _size = fut.result()
            top_up()
            if pending and (pending[0][1].shape != arr.shape or len(pending) >= batch_size):
                run_batch(pending)
                pending = []
            pending.append((path, arr))
        if pending:
            run_batch(pending)
        for fut in futures:
            if fut is not None:
                fut.result()
    finally:
        decoders.shutdown(wait=True)
        writers.shutdown(wait=True)


def enhance_batch_images(input_dir, output_dir, device, max_size=None, enable_multi_scale=False,
                         enable_content_aware=False, batch_size=16, model=None, decode_workers=None, encode_workers=None, amp=None):
    device = resolve_device(device)
    amp_context(amp)   # an unknown amp fails before any file is read
    print("正在加载模型...")
    if model is None:
        model = UP_Retinex().to(device).eval()
    files = list_images(input_dir)
    if not files:
        print(f"在目录 '{input_dir}' 中未找到有效图像文件")
        return
    mine = shard_for_rank(files)
    print(f"找到 {len(files)} 个图像文件 (本进程处理 {len(mine)} 个)")
    t0 = time.time()

    def write_files(stem, low8, enh8, illu8):
        save_image(enh8, os.path.join(output_dir, f"{stem}_enhanced.png"))
        save_image(illu8, os.path.join(output_dir, f"{stem}_illumination.png"))
        create_comparison(low8, enh8, os.path.join(output_dir, f"{stem}_comparison.png"))

    def host_fn(path, arr):      # host tensors: the reference's own behaviour, one by one (the hot-path ops will refuse them)
        low = torch.from_numpy(arr).permute(2, 0, 1).to(torch.float32).div(255.0).unsqueeze(0)
        if max_size is not None:
            low = letterbox_tensor(low[0], new_shape=max_size, auto=True, scaleup=False)[0].unsqueeze(0)
        with amp_context(amp):
            enhanced, illu = _enhance_tensor(model, low, device, enable_multi_scale, enable_content_aware)
        _write_outputs(low, enhanced, illu, path, output_dir)

    def frame_fn(low):
        with amp_context(amp):   # entered by the thread that runs the batch (autocast state is per thread)
            return enhance_frames_u8(model, low, enable_multi_scale, enable_content_aware)

    run_batch_pipeline(mine, output_dir, device, max_size, batch_size, frame_fn, write_files, host_fn, decode_workers,
                       encode_workers)
    total = time.time() - t0
    print("=" * 50)
    print(f"总共处理了 {len(mine)} 张图像")
    print(f"总耗时: {total:.2f}s")
    if mine:
        print(f"平均每张图像耗时: {total / len(mine):.4f}s")
    print("=" * 50)
