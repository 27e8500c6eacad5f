"""ctypes binding of libupretinex_b200.so (C ABI: include/upretinex_b200.h) + tensor-level wrappers.

PyTorch is plumbing here (device memory, streams); every op is one call into the C ABI with raw
device pointers and the current CUDA stream.  Missing library or missing GPU -> exception; there
is deliberately no fallback path.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Optional, Tuple

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libupretinex_b200.so")

_lib = None
_lock = threading.Lock()

STATUS = {0: "UPR_OK", -1: "UPR_E_NULL", -2: "UPR_E_SHAPE", -3: "UPR_E_WORKSPACE", -4: "UPR_E_PARAM",
          -5: "UPR_E_DEVICE"}


class UprError(RuntimeError):
    def __init__(self, status: int, what: str):
        self.status = status
        super().__init__(f"{what} failed: status {status} ({status_string(status)})")


def _declare(lib):
    vp, i32, f64, sz = C.c_void_p, C.c_int, C.c_double, C.c_size_t
    lib.upr_version.restype = C.c_char_p
    lib.upr_status_string.restype = C.c_char_p
    lib.upr_status_string.argtypes = [i32]
    lib.upr_device_check.restype = i32
    lib.upr_clahe_workspace_bytes.restype = sz
    lib.upr_clahe_workspace_bytes.argtypes = [i32] * 5
    lib.upr_clahe_lab_f32.restype = i32
    lib.upr_clahe_lab_f32.argtypes = [vp, vp, i32, i32, i32, f64, i32, i32, vp, sz, vp]
    lib.upr_clahe_lab_u8.restype = i32
    lib.upr_clahe_lab_u8.argtypes = [vp, vp, i32, i32, i32, f64, i32, i32, vp, sz, vp]
    lib.upr_clahe_lab_f32_u8.restype = i32
    lib.upr_clahe_lab_f32_u8.argtypes = [vp, vp, i32, i32, i32, f64, i32, i32, vp, sz, vp]
    lib.upr_retinex_clahe_f32.restype = i32
    lib.upr_retinex_clahe_f32.argtypes = [vp, vp, vp, vp, i32, i32, i32, C.c_float, f64, i32, i32, vp, sz, vp]
    lib.upr_retinex_clahe_f32_u8.restype = i32
    lib.upr_retinex_clahe_f32_u8.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, C.c_float, f64, i32, i32, vp, sz, vp]
    lib.upr_clahe_lab_stages_f32.restype = i32
    lib.upr_clahe_lab_stages_f32.argtypes = [vp, vp, i32, i32, i32, f64, i32, i32, vp, sz, i32, vp]
    lib.upr_clahe_debug_dump.restype = i32
    lib.upr_clahe_debug_dump.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, vp, vp]
    lib.upr_clahe_debug_load.restype = i32
    lib.upr_clahe_debug_load.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, vp]
    lib.upr_get_tables.restype = i32
    lib.upr_get_tables.argtypes = [vp] * 4
    f32 = C.c_float
    lib.upr_clahe_lab_f32_host.restype = i32
    lib.upr_clahe_lab_f32_host.argtypes = [vp, vp, i32, i32, i32, f64, i32, i32, i32]
    lib.upr_clahe_lab_u8_host.restype = i32
    lib.upr_clahe_lab_u8_host.argtypes = [vp, vp, i32, i32, i32, f64, i32, i32, i32]
    lib.upr_host_pool_release.restype = i32
    lib.upr_brightness_hist_f32.restype = i32
    lib.upr_brightness_hist_f32.argtypes = [vp, i32, i32, i32, vp, vp]
    lib.upr_multiscale_workspace_bytes.restype = sz
    lib.upr_multiscale_workspace_bytes.argtypes = [i32] * 3
    lib.upr_multiscale_stats_f32.restype = i32
    lib.upr_multiscale_stats_f32.argtypes = [vp, i32, i32, i32, vp, vp, vp, sz, i32, vp]
    lib.upr_multiscale_features_f32.restype = i32
    lib.upr_multiscale_features_f32.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, sz, vp]
    lib.upr_scale_clamp_f32.restype = i32
    lib.upr_scale_clamp_f32.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
    lib.upr_saliency_workspace_bytes.restype = sz
    lib.upr_saliency_workspace_bytes.argtypes = [i32] * 3
    lib.upr_saliency_f32.restype = i32
    lib.upr_saliency_f32.argtypes = [vp, i32, i32, i32, vp, vp, sz, vp]
    lib.upr_attention_f32.restype = i32
    lib.upr_attention_f32.argtypes = [vp, i32, i32, i32, vp, vp, sz, vp]
    lib.upr_attention_apply_f32.restype = i32
    lib.upr_attention_apply_f32.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
    lib.upr_content_aware_apply_f32.restype = i32
    lib.upr_content_aware_apply_f32.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, sz, vp]
    lib.upr_quantize_u8_f32.restype = i32
    lib.upr_quantize_u8_f32.argtypes = [vp, vp, i32, i32, i32, i32, vp]
    lib.upr_multiscale_enhance_f32.restype = i32
    lib.upr_multiscale_enhance_f32.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, vp, sz, vp]
    lib.upr_content_multiscale_f32.restype = i32
    lib.upr_content_multiscale_f32.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, sz, vp, sz, vp]
    lib.upr_content_multiscale_apply_f32.restype = i32
    lib.upr_content_multiscale_apply_f32.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, vp, sz, vp]
    lib.upr_retinex_recombine_f32.restype = i32
    lib.upr_retinex_recombine_f32.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, f32, vp]
    lib.upr_retinex_decompose_f32.restype = i32
    lib.upr_retinex_decompose_f32.argtypes = [vp, vp, vp, i32, i32, i32, f32, vp]
    lib.upr_letterbox_f32.restype = i32
    lib.upr_letterbox_f32.argtypes = [vp, vp] + [i32] * 10 + [vp, vp]
    lib.upr_letterbox_u8_f32.restype = i32
    lib.upr_letterbox_u8_f32.argtypes = [vp, vp] + [i32] * 10 + [vp, vp]
    lib.upr_texture_workspace_bytes.restype = sz
    lib.upr_texture_workspace_bytes.argtypes = [i32]
    lib.upr_texture_workspace_init.restype = i32
    lib.upr_texture_workspace_init.argtypes = [vp, sz, i32, vp]
    lib.upr_texture_tv_f32.restype = i32
    lib.upr_texture_tv_f32.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp, sz, vp]
    lib.upr_texture_edge_density_f32.restype = i32
    lib.upr_texture_edge_density_f32.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp, sz, vp]
    lib.upr_enh_losses_workspace_bytes.restype = sz
    lib.upr_enh_losses_workspace_bytes.argtypes = [i32]
    lib.upr_enh_losses_saved_floats.restype = sz
    lib.upr_enh_losses_saved_floats.argtypes = [i32] * 4
    lib.upr_enh_losses_f32.restype = i32
    lib.upr_enh_losses_f32.argtypes = [vp, vp, i32, i32, i32, f64, i32, vp, vp, vp, sz, vp]
    lib.upr_enh_losses_grad_f32.restype = i32
    lib.upr_enh_losses_grad_f32.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, vp, vp]
    lib.upr_smooth_loss_workspace_bytes.restype = sz
    lib.upr_smooth_loss_workspace_bytes.argtypes = [i32] * 3
    lib.upr_edge_smooth_loss_f32.restype = i32
    lib.upr_edge_smooth_loss_f32.argtypes = [vp, vp, i32, i32, i32, i32, i32, f32, f32, vp, vp, vp, sz, vp]
    lib.upr_peer_stats_buffer_bytes.restype = sz
    lib.upr_peer_set_timeout_ms.restype = i32
    lib.upr_peer_set_timeout_ms.argtypes = [f64]
    lib.upr_peer_status.restype = i32
    lib.upr_peer_status.argtypes = [vp, vp, vp]
    lib.upr_texture_weight_peer_f32.restype = i32
    lib.upr_texture_weight_peer_f32.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, vp, sz, vp, i32, i32, C.c_uint, f32, vp, vp]
    lib.upr_dynamic_smooth_weight_f32.restype = i32
    lib.upr_dynamic_smooth_weight_f32.argtypes = [vp, f32, vp, vp]
    lib.upr_ext_gaussian_blur_f32.restype = i32
    lib.upr_ext_gaussian_blur_f32.argtypes = [vp, vp, i32, i32, i32, i32, f64, vp]
    lib.upr_ext_msr_f32.restype = i32
    lib.upr_ext_msr_f32.argtypes = [vp, vp, i32, i32, i32, i32, C.POINTER(C.c_int), C.POINTER(C.c_double), C.POINTER(C.c_float),
                                    f32, vp]
    lib.upr_ext_pyr_down_f32.restype = i32
    lib.upr_ext_pyr_down_f32.argtypes = [vp, vp, i32, i32, i32, vp]
    lib.upr_ext_gamma_f32.restype = i32
    lib.upr_ext_gamma_f32.argtypes = [vp, vp, C.c_longlong, f32, vp]


def lib():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(nvcc, sm_100a).  upretinex-b200 has no CPU fallback.")
                handle = C.CDLL(LIB_PATH)
                _declare(handle)
                _lib = handle
    return _lib


def bind_to_gpu_numa_node(device_index: int) -> bool:
    """One process per GPU: pin this process to the CPU cores next to ``device_index`` (NVML's ideal CPU affinity), so that
    the pinned host buffers it allocates afterwards are first-touched on the GPU's own NUMA node.  With eight ranks moving
    12 + 12 bytes per pixel over PCIe the host side is the bottleneck, and remote-node buffers cross the socket link twice.
    Call it before allocating host memory or starting worker threads.  Returns False if NVML is unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(int(device_index)))
        return True
    except Exception:
        return False


def status_string(status: int) -> str:
    if status <= 0:
        return STATUS.get(status, "UPR_E_?")
    try:
        return lib().upr_status_string(status).decode()
    except Exception:  # pragma: no cover
        return f"cudaError {status}"


def check(status: int, what: str) -> None:
    if status != 0:
        raise UprError(status, what)


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


class _NoSwitch:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_NO_SWITCH = _NoSwitch()


def _dev(device):
    """Context that makes `device` current for a call; nothing to do (and ~4 us of Python saved per call) when it already is."""
    idx = device.index if isinstance(device, torch.device) else torch.device(device).index
    if idx is None or idx == torch.cuda.current_device():
        return _NO_SWITCH
    return torch.cuda.device(idx)


def _cuda(t: torch.Tensor, name: str, dtype: torch.dtype = torch.float32, shape=None, device=None) -> torch.Tensor:
    """`t` made contiguous, after checks that cost attribute reads only: RuntimeError off the GPU, TypeError for another dtype,
    ValueError for another shape (None in `shape` = any size) or for a device other than `device`."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must live on a CUDA device (upretinex-b200 has no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if shape is not None and (t.dim() != len(shape) or any(s is not None and s != d for s, d in zip(shape, t.shape))):
        raise ValueError(f"{name} must have shape {tuple('*' if s is None else s for s in shape)}, got {tuple(t.shape)}")
    if device is not None and t.device != device:
        raise ValueError(f"{name} is on {t.device}, the call's first tensor on {device}")
    return t.contiguous()


def _out(out: Optional[torch.Tensor], shape, dtype: torch.dtype, device: torch.device) -> torch.Tensor:
    """A new tensor when `out` is None; otherwise `out`, which must be contiguous with exactly this shape, dtype and device
    (ValueError).  Whether it may alias an input is for the entry point to decide."""
    if out is None:
        return torch.empty(shape, dtype=dtype, device=device)
    if not (isinstance(out, torch.Tensor) and out.shape == shape and out.dtype == dtype and out.device == device
            and out.is_contiguous()):
        raise ValueError(f"out must be a contiguous {dtype} tensor of shape {tuple(shape)} on {device}")
    return out


def _ws(size_fn: str, size_args, device: torch.device, zero_tag: Optional[str] = None) -> torch.Tensor:
    """The workspace that the size function `size_fn` asks for: workspace(), or zero_workspace(zero_tag, ...) for the kernels
    that need it zero-filled.  Size 0 means the entry point would reject the shape: UprError(UPR_E_SHAPE).  Call it with
    `device` current: the workspace belongs to that device's current stream."""
    nbytes = getattr(lib(), size_fn)(*size_args)
    if nbytes == 0:
        raise UprError(-2, size_fn)
    return workspace(nbytes, device) if zero_tag is None else zero_workspace(zero_tag, nbytes, device)


def _run(entry: str, *args) -> None:
    """Call the entry point `entry` with `args` and the current stream; UprError for a failed status."""
    check(getattr(lib(), entry)(*args, _stream()), entry)


# one growing workspace per (device, stream): the C ABI never allocates
_workspaces = {}


def workspace(nbytes: int, device: torch.device) -> torch.Tensor:
    key = (device.index if device.index is not None else torch.cuda.current_device(), _stream())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


_zero_ws = {}


def zero_workspace(tag: str, nbytes: int, device: torch.device) -> torch.Tensor:
    """Workspace that is zero-filled when (re)allocated; the ticket kernels leave it clean."""
    key = (tag, device.index if device.index is not None else torch.cuda.current_device(), _stream())
    ws = _zero_ws.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.zeros(max(nbytes, 1), dtype=torch.uint8, device=device)
        _zero_ws[key] = ws
    return ws


def release_workspaces() -> None:
    _workspaces.clear()
    _zero_ws.clear()


# ------------------------------------------------------------------------------------------------
# a1: CLAHE in Lab
# ------------------------------------------------------------------------------------------------
def _clahe(entry: str, x: torch.Tensor, clip_limit: float, tiles: Tuple[int, int], out: Optional[torch.Tensor],
           u8_in: bool = False, u8_out: bool = False, retinex=None, extra=()) -> torch.Tensor:
    """The body of the CLAHE family.  x: [N,3,H,W] f32, or with u8_in [N,H,W,3] uint8 (packed RGB); out: [N,3,H,W] f32, or
    with u8_out [N,H,W,3] uint8.  retinex = (illu, e, eps): CLAHE of the Retinex recombination of x, e and illu (the
    upr_retinex_clahe_* entries).  extra: arguments of `entry` between the workspace and the stream."""
    if u8_in:
        x = _cuda(x, "x", torch.uint8)
        if x.dim() != 4 or x.shape[3] != 3:      # a planar u8 tensor is not the decoded file this entry reads
            raise TypeError(f"expected uint8 [N,H,W,3], got {tuple(x.shape)}")
        n, h, w, _ = x.shape
    else:
        x = _cuda(x, "x", shape=(None, 3, None, None))
        n, _, h, w = x.shape
    dev = x.device
    out = _out(out, (n, h, w, 3), torch.uint8, dev) if u8_out else _out(out, x.shape, torch.float32, dev)
    if retinex is not None:
        illu, e, eps = retinex
        illu = _cuda(illu, "illu", device=dev)
        e = _cuda(e, "e", shape=x.shape, device=dev)
        if illu.numel() != n * h * w:
            raise ValueError(f"illu must be [N,1,H,W], got {tuple(illu.shape)}")
    tx, ty = int(tiles[0]), int(tiles[1])
    with _dev(dev):
        ws = _ws("upr_clahe_workspace_bytes", (n, h, w, tx, ty), dev)
        tail = (float(clip_limit), tx, ty, ws.data_ptr(), ws.numel(), *extra)
        if retinex is None:
            _run(entry, x.data_ptr(), out.data_ptr(), n, h, w, *tail)
        elif not u8_out:
            _run(entry, x.data_ptr(), illu.data_ptr(), e.data_ptr(), out.data_ptr(), n, h, w, float(eps), *tail)
        else:
            fn = getattr(lib(), entry)
            ptrs = (x.data_ptr(), illu.data_ptr(), e.data_ptr(), out.data_ptr())
            args = (n, h, w, float(eps), *tail, _stream())
            rc = fn(*ptrs, None, *args)
            if rc == -3:   # ragged shape: the recombination needs a scratch frame
                scratch = torch.empty_like(x)
                rc = fn(*ptrs, scratch.data_ptr(), *args)
            check(rc, entry)
    return out


def clahe_lab(x: torch.Tensor, clip_limit: float = 2.0, tiles: Tuple[int, int] = (8, 8),
              out: Optional[torch.Tensor] = None, stage_mask: int = 3) -> torch.Tensor:
    """x: [N,3,H,W] f32 CUDA -> [N,3,H,W] f32 CUDA (upr_clahe_lab_f32).  stage_mask != 3 is the profiling
    hook upr_clahe_lab_stages_f32 (only meaningful right after a full call with the same arguments)."""
    if stage_mask == 3:
        return _clahe("upr_clahe_lab_f32", x, clip_limit, tiles, out)
    return _clahe("upr_clahe_lab_stages_f32", x, clip_limit, tiles, out, extra=(int(stage_mask),))


def clahe_lab_u8(x: torch.Tensor, clip_limit: float = 2.0, tiles: Tuple[int, int] = (8, 8),
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x: [N,H,W,3] uint8 CUDA (packed RGB, what an image file decodes to) -> [N,H,W,3] uint8 CUDA (upr_clahe_lab_u8)."""
    return _clahe("upr_clahe_lab_u8", x, clip_limit, tiles, out, u8_in=True, u8_out=True)


def clahe_lab_f32_u8(x: torch.Tensor, clip_limit: float = 2.0, tiles: Tuple[int, int] = (8, 8),
                     out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x: [N,3,H,W] f32 CUDA -> [N,H,W,3] uint8 CUDA: upr_clahe_lab_f32 followed by the quantisation of save_image, in one op."""
    return _clahe("upr_clahe_lab_f32_u8", x, clip_limit, tiles, out, u8_out=True)


def clahe_debug(x_shape, tiles: Tuple[int, int] = (8, 8), device=None, want_lab: bool = True):
    """Histograms / LUTs / Lab intermediate of the last clahe_lab() call on this stream."""
    n, _, h, w = x_shape
    tx, ty = int(tiles[0]), int(tiles[1])
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    L = lib()
    with _dev(device):
        ws = workspace(L.upr_clahe_workspace_bytes(n, h, w, tx, ty), device)
        hist = torch.empty((n, ty * tx, 256), dtype=torch.int32, device=device)
        lut = torch.empty((n, ty * tx, 256), dtype=torch.uint8, device=device)
        lab = torch.empty((n, 3, h, w), dtype=torch.uint8, device=device) if want_lab else None
        check(L.upr_clahe_debug_dump(ws.data_ptr(), n, h, w, tx, ty, hist.data_ptr(), lut.data_ptr(),
                                     lab.data_ptr() if lab is not None else None, _stream()), "upr_clahe_debug_dump")
    return hist, lut, lab


def clahe_map_only(lab_u8: torch.Tensor, lut_u8: torch.Tensor, tiles: Tuple[int, int] = (8, 8)) -> torch.Tensor:
    """The map stage of clahe_lab() alone on chosen inputs: lab_u8 [N,3,H,W] uint8 (L, a, b planes) and lut_u8
    [N,ty*tx,256] uint8 (one LUT per tile) -> [N,3,H,W] f32, the de-quantised sRGB of (bilinear LUT interpolation of L, a, b).
    Loads both into the workspace (upr_clahe_debug_load) and runs upr_clahe_lab_stages_f32 with stage_mask = 2."""
    lab_u8 = _cuda(lab_u8, "lab_u8", torch.uint8, shape=(None, 3, None, None))
    n, _, h, w = lab_u8.shape
    tx, ty = int(tiles[0]), int(tiles[1])
    dev = lab_u8.device
    lut_u8 = _cuda(lut_u8, "lut_u8", torch.uint8, shape=(n, ty * tx, 256), device=dev)
    out = _out(None, lab_u8.shape, torch.float32, dev)
    with _dev(dev):
        ws = _ws("upr_clahe_workspace_bytes", (n, h, w, tx, ty), dev)
        _run("upr_clahe_debug_load", ws.data_ptr(), n, h, w, tx, ty, lut_u8.data_ptr(), lab_u8.data_ptr())
        # the stages entry checks its input pointer although the map stage does not read it: pass the output
        _run("upr_clahe_lab_stages_f32", out.data_ptr(), out.data_ptr(), n, h, w, 2.0, tx, ty, ws.data_ptr(), ws.numel(), 2)
    return out


def tables():
    import numpy as np
    g = np.zeros(256, np.uint16); c = np.zeros(2048, np.uint16)
    yf = np.zeros(256, np.uint32); ig = np.zeros(4096, np.uint8)
    check(lib().upr_get_tables(g.ctypes.data, c.ctypes.data, yf.ctypes.data, ig.ctypes.data), "upr_get_tables")
    return {"gamma": g, "cbrt": c, "ify": (yf & 0xFFFF).astype(np.uint16), "y": (yf >> 16).astype(np.uint16),
            "invgamma": ig}


def _clahe_host(entry: str, x: torch.Tensor, clip_limit: float, tiles: Tuple[int, int], out: Optional[torch.Tensor],
                frames_per_chunk: int, u8: bool) -> torch.Tensor:
    """The body of the two host entries: x and out host tensors, [N,3,H,W] f32, or with u8 [N,H,W,3] uint8 (packed RGB)."""
    dtype = torch.uint8 if u8 else torch.float32
    if x.is_cuda or x.dtype != dtype:
        raise TypeError(f"{entry} expects a {dtype} host tensor")
    if x.dim() != 4 or x.shape[3 if u8 else 1] != 3:
        raise ValueError(f"expected {'[N,H,W,3]' if u8 else '[N,3,H,W]'}, got {tuple(x.shape)}")
    if not torch.cuda.is_available():
        raise RuntimeError("no CUDA device: upretinex-b200 has no CPU path")
    x = x.contiguous()
    n, h, w = x.shape[:3] if u8 else (x.shape[0], x.shape[2], x.shape[3])
    if out is None:
        out = torch.empty(x.shape, dtype=dtype, pin_memory=True)
    elif out.is_cuda or out.shape != x.shape or out.dtype != dtype or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous {dtype} host tensor shaped like x")
    check(getattr(lib(), entry)(x.data_ptr(), out.data_ptr(), n, h, w, float(clip_limit), int(tiles[0]), int(tiles[1]),
                                int(frames_per_chunk)), entry)
    return out


def clahe_lab_host(x: torch.Tensor, clip_limit: float = 2.0, tiles: Tuple[int, int] = (8, 8),
                   out: Optional[torch.Tensor] = None, frames_per_chunk: int = 0) -> torch.Tensor:
    """x: [N,3,H,W] f32 HOST tensor -> [N,3,H,W] f32 HOST (pinned) tensor (upr_clahe_lab_f32_host).

    H2D, kernels and D2H are pipelined inside the library; pin ``x`` for full PCIe speed."""
    return _clahe_host("upr_clahe_lab_f32_host", x, clip_limit, tiles, out, frames_per_chunk, u8=False)


def clahe_lab_u8_host(x: torch.Tensor, clip_limit: float = 2.0, tiles: Tuple[int, int] = (8, 8),
                      out: Optional[torch.Tensor] = None, frames_per_chunk: int = 0) -> torch.Tensor:
    """x: [N,H,W,3] uint8 HOST tensor (decoded image files) -> [N,H,W,3] uint8 HOST (pinned) tensor (upr_clahe_lab_u8_host)."""
    return _clahe_host("upr_clahe_lab_u8_host", x, clip_limit, tiles, out, frames_per_chunk, u8=True)


# ------------------------------------------------------------------------------------------------
# a3: brightness histogram
# ------------------------------------------------------------------------------------------------
def brightness_hist(x: torch.Tensor) -> torch.Tensor:
    """x: [N,3,H,W] f32 CUDA -> [N,256] int32 CUDA histogram of the u8 gray image."""
    x = _cuda(x, "x", shape=(None, 3, None, None))
    n, _, h, w = x.shape
    hist = torch.empty((n, 256), dtype=torch.int32, device=x.device)
    with _dev(x.device):
        _run("upr_brightness_hist_f32", x.data_ptr(), n, h, w, hist.data_ptr())
    return hist


# ------------------------------------------------------------------------------------------------
# a4/a5: multi-scale statistics
# ------------------------------------------------------------------------------------------------
def multiscale_stats(x: torch.Tensor, force_generic: bool = False):
    """x: [N,3,H,W] -> (means [N,3] f32, gain [N] f32), both on the device (no host sync)."""
    x = _cuda(x, "x", shape=(None, 3, None, None))
    n, _, h, w = x.shape
    if int(h * 0.25) < 1 or int(w * 0.25) < 1:
        raise ValueError("image too small for the 1/4 scale")
    means = torch.empty((n, 3), dtype=torch.float32, device=x.device)
    gain = torch.empty((n,), dtype=torch.float32, device=x.device)
    with _dev(x.device):
        ws = _ws("upr_multiscale_workspace_bytes", (n, h, w), x.device, "ms")
        _run("upr_multiscale_stats_f32", x.data_ptr(), n, h, w, means.data_ptr(), gain.data_ptr(), ws.data_ptr(), ws.numel(),
             1 if force_generic else 0)
    return means, gain


def multiscale_enhance(x: torch.Tensor, enh: torch.Tensor, out: torch.Tensor | None = None):
    """a4 + a5 in one call: out = clamp(enh * gain(x)[frame], 0, 1) -> (out, means [N,3], gain [N]); large batches run chunk by
    chunk on two library-owned side streams (upr_multiscale_enhance_f32).  out may be enh."""
    x = _cuda(x, "x", shape=(None, 3, None, None))
    enh = _cuda(enh, "enh", shape=x.shape, device=x.device)
    n, _, h, w = x.shape
    if int(h * 0.25) < 1 or int(w * 0.25) < 1:
        raise ValueError("image too small for the 1/4 scale")
    out = _out(out, x.shape, torch.float32, x.device)
    means = torch.empty((n, 3), dtype=torch.float32, device=x.device)
    gain = torch.empty((n,), dtype=torch.float32, device=x.device)
    with _dev(x.device):
        ws = _ws("upr_multiscale_workspace_bytes", (n, h, w), x.device, "ms")
        _run("upr_multiscale_enhance_f32", x.data_ptr(), enh.data_ptr(), out.data_ptr(), means.data_ptr(), gain.data_ptr(), n, h, w,
             ws.data_ptr(), ws.numel())
    return out, means, gain


def multiscale_features(x: torch.Tensor):
    """x: [N,3,H,W] -> ([N,7,H,W], [N,7,H/2,W/2], [N,7,H/4,W/4], means [N,3], gain [N])."""
    x = _cuda(x, "x", shape=(None, 3, None, None))
    n, _, h, w = x.shape
    h2, w2, h4, w4 = int(h * 0.5), int(w * 0.5), int(h * 0.25), int(w * 0.25)
    if h4 < 1 or w4 < 1:
        raise ValueError("image too small for the 1/4 scale")
    f1 = torch.empty((n, 7, h, w), dtype=torch.float32, device=x.device)
    f2 = torch.empty((n, 7, h2, w2), dtype=torch.float32, device=x.device)
    f3 = torch.empty((n, 7, h4, w4), dtype=torch.float32, device=x.device)
    means = torch.empty((n, 3), dtype=torch.float32, device=x.device)
    gain = torch.empty((n,), dtype=torch.float32, device=x.device)
    with _dev(x.device):
        ws = _ws("upr_multiscale_workspace_bytes", (n, h, w), x.device, "ms")
        _run("upr_multiscale_features_f32", x.data_ptr(), n, h, w, f1.data_ptr(), f2.data_ptr(), f3.data_ptr(), means.data_ptr(),
             gain.data_ptr(), ws.data_ptr(), ws.numel())
    return f1, f2, f3, means, gain


def scale_clamp(enh: torch.Tensor, gain: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """clamp(enh * gain[image], 0, 1); enh [N,C,H,W], gain [N] f32 on the same device."""
    enh = _cuda(enh, "enh")
    gain = _cuda(gain, "gain", device=enh.device).reshape(-1)
    n, c, h, w = enh.shape
    if gain.numel() != n:
        raise ValueError("gain must have one entry per image")
    out = _out(out, enh.shape, torch.float32, enh.device)
    with _dev(enh.device):
        _run("upr_scale_clamp_f32", enh.data_ptr(), gain.data_ptr(), out.data_ptr(), n, c, h, w)
    return out


def retinex_clahe(x: torch.Tensor, illu: torch.Tensor, e: torch.Tensor, clip_limit: float = 2.0,
                  tiles: Tuple[int, int] = (8, 8), eps: float = 1e-6, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """CLAHE-in-Lab of the Retinex recombination R*e + (1-R)*e^2, R = x/(illu+eps), in one call (upr_retinex_clahe_f32):
    the recombined frame is never materialised.  Bit-identical to retinex_recombine(...)[1] -> clahe_lab(...)."""
    return _clahe("upr_retinex_clahe_f32", x, clip_limit, tiles, out, retinex=(illu, e, eps))


def retinex_clahe_u8(x: torch.Tensor, illu: torch.Tensor, e: torch.Tensor, clip_limit: float = 2.0,
                     tiles: Tuple[int, int] = (8, 8), eps: float = 1e-6, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """retinex_clahe() emitting the packed u8 RGB frame [N,H,W,3] that save_image would store (upr_retinex_clahe_f32_u8)."""
    return _clahe("upr_retinex_clahe_f32_u8", x, clip_limit, tiles, out, u8_out=True, retinex=(illu, e, eps))


# ------------------------------------------------------------------------------------------------
# a6/a7: saliency / attention
# ------------------------------------------------------------------------------------------------
def _sal(fn_name: str, x: torch.Tensor) -> torch.Tensor:
    x = _cuda(x, "x", shape=(None, 3, None, None))
    n, _, h, w = x.shape
    out = torch.empty((n, 1, h, w), dtype=torch.float32, device=x.device)
    with _dev(x.device):
        ws = _ws("upr_saliency_workspace_bytes", (n, h, w), x.device)
        _run(fn_name, x.data_ptr(), n, h, w, out.data_ptr(), ws.data_ptr(), ws.numel())
    return out


def saliency(x: torch.Tensor) -> torch.Tensor:
    return _sal("upr_saliency_f32", x)


def attention(x: torch.Tensor) -> torch.Tensor:
    return _sal("upr_attention_f32", x)


def attention_apply(enh: torch.Tensor, att: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    enh = _cuda(enh, "enh")
    att = _cuda(att, "att", device=enh.device)
    n, c, h, w = enh.shape
    if att.numel() != n * h * w:
        raise ValueError("att must be [N,1,H,W]")
    out = _out(out, enh.shape, torch.float32, enh.device)
    with _dev(enh.device):
        _run("upr_attention_apply_f32", enh.data_ptr(), att.data_ptr(), out.data_ptr(), n, c, h, w)
    return out


# ------------------------------------------------------------------------------------------------
# a8: Retinex decomposition / recombination
# ------------------------------------------------------------------------------------------------
def content_aware_apply(x: torch.Tensor, enh: torch.Tensor, out: Optional[torch.Tensor] = None, want_attention: bool = False):
    """clamp(enh * (1 + 0.2 * attention(x)), 0, 1) in three passes (upr_content_aware_apply_f32); returns out, or
    (out, attention) with want_attention.  Identical to attention() followed by attention_apply()."""
    x = _cuda(x, "x", shape=(None, 3, None, None))
    enh = _cuda(enh, "enh", shape=x.shape, device=x.device)
    n, _, h, w = x.shape
    out = _out(out, x.shape, torch.float32, x.device)
    att = torch.empty((n, 1, h, w), dtype=torch.float32, device=x.device) if want_attention else None
    with _dev(x.device):
        ws = _ws("upr_saliency_workspace_bytes", (n, h, w), x.device)
        _run("upr_content_aware_apply_f32", x.data_ptr(), enh.data_ptr(), out.data_ptr(), att.data_ptr() if att is not None else None,
             n, h, w, ws.data_ptr(), ws.numel())
    return (out, att) if want_attention else out


def content_multiscale_apply(x: torch.Tensor, enh: torch.Tensor, out: Optional[torch.Tensor] = None, gain: Optional[torch.Tensor] = None):
    """BASELINE config 5 chain in four launches: multi-scale statistics of x (gain stays on the device), saliency blur, raw
    attention, and ONE epilogue  clamp(clamp(enh * (1 + 0.2 att), 0, 1) * gain, 0, 1)  (upr_content_multiscale_apply_f32).
    Equal to content_aware_apply() followed by scale_clamp().  Returns (out, gain [N])."""
    x = _cuda(x, "x", shape=(None, 3, None, None))
    enh = _cuda(enh, "enh", shape=x.shape, device=x.device)
    n, _, h, w = x.shape
    out = _out(out, x.shape, torch.float32, x.device)
    if gain is None:
        # statistics inside the chunk schedule of the content-aware passes (upr_content_multiscale_f32)
        if int(h * 0.25) < 1 or int(w * 0.25) < 1:
            raise ValueError("image too small for the 1/4 scale")
        means = torch.empty((n, 3), dtype=torch.float32, device=x.device)
        gain = torch.empty((n,), dtype=torch.float32, device=x.device)
        with _dev(x.device):
            ws = _ws("upr_saliency_workspace_bytes", (n, h, w), x.device)
            ms_ws = _ws("upr_multiscale_workspace_bytes", (n, h, w), x.device, "ms")
            _run("upr_content_multiscale_f32", x.data_ptr(), enh.data_ptr(), out.data_ptr(), None, means.data_ptr(), gain.data_ptr(),
                 n, h, w, ws.data_ptr(), ws.numel(), ms_ws.data_ptr(), ms_ws.numel())
        return out, gain
    gain = _cuda(gain, "gain", device=x.device).reshape(-1)
    if gain.numel() != n:
        raise ValueError("gain must have one entry per image")
    with _dev(x.device):
        ws = _ws("upr_saliency_workspace_bytes", (n, h, w), x.device)
        _run("upr_content_multiscale_apply_f32", x.data_ptr(), enh.data_ptr(), gain.data_ptr(), out.data_ptr(), None, n, h, w,
             ws.data_ptr(), ws.numel())
    return out, gain


def retinex_recombine(x: torch.Tensor, illu: torch.Tensor, e: torch.Tensor, want_reflectance: bool = True,
                      eps: float = 1e-6):
    """(reflectance | None, enhanced) for x,e [N,3,H,W] and illu [N,1,H,W]."""
    x = _cuda(x, "x", shape=(None, 3, None, None))
    illu = _cuda(illu, "illu", device=x.device)
    e = _cuda(e, "e", shape=x.shape, device=x.device)
    n, _, h, w = x.shape
    if illu.numel() != n * h * w:
        raise ValueError(f"illu must be [N,1,H,W], got {tuple(illu.shape)}")
    refl = torch.empty_like(x) if want_reflectance else None
    enh = torch.empty_like(x)
    with _dev(x.device):
        _run("upr_retinex_recombine_f32", x.data_ptr(), illu.data_ptr(), e.data_ptr(), refl.data_ptr() if refl is not None else None,
             enh.data_ptr(), n, h, w, float(eps))
    return refl, enh


def quantize_u8(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """save_image's (clip(x, 0, 1) * 255).astype(uint8) on the device: [N,C,H,W] f32 (C = 1 or 3) -> [N,H,W,C] u8."""
    x = _cuda(x, "x")
    n, c, h, w = x.shape
    if c not in (1, 3):
        raise ValueError("expected 1 or 3 channels")
    out = _out(out, (n, h, w, c), torch.uint8, x.device)
    with _dev(x.device):
        _run("upr_quantize_u8_f32", x.data_ptr(), out.data_ptr(), n, c, h, w)
    return out


def retinex_decompose(x: torch.Tensor, illu: torch.Tensor, eps: float = 1e-6) -> torch.Tensor:
    x = _cuda(x, "x", shape=(None, 3, None, None))
    illu = _cuda(illu, "illu", device=x.device)
    n, _, h, w = x.shape
    if illu.numel() != n * h * w:
        raise ValueError(f"illu must be [N,1,H,W], got {tuple(illu.shape)}")
    refl = torch.empty_like(x)
    with _dev(x.device):
        _run("upr_retinex_decompose_f32", x.data_ptr(), illu.data_ptr(), refl.data_ptr(), n, h, w, float(eps))
    return refl


# ------------------------------------------------------------------------------------------------
# a9/a10: texture complexity, dynamic smoothness weight
# ------------------------------------------------------------------------------------------------
def texture_complexity(x: torch.Tensor, method: str = "tv", want_batch_stats: bool = False):
    """x: [B,C,H,W] f32 CUDA -> per-image complexity [B] (and [sum, B] if want_batch_stats)."""
    if method not in ("tv", "edge_density"):
        raise ValueError(f"unsupported texture complexity method: {method}")
    x = _cuda(x, "x")
    b, c, h, w = x.shape
    out = torch.empty((b,), dtype=torch.float32, device=x.device)
    stats = torch.empty((2,), dtype=torch.float32, device=x.device) if want_batch_stats else None
    with _dev(x.device):
        ws = _ws("upr_texture_workspace_bytes", (b,), x.device, "tex")
        _run(f"upr_texture_{method}_f32", x.data_ptr(), b, c, h, w, out.data_ptr(), stats.data_ptr() if stats is not None else None,
             ws.data_ptr(), ws.numel())
    return (out, stats) if want_batch_stats else out


def _saved_floats(b: int, h: int, w: int, patch: int) -> int:
    nsaved = lib().upr_enh_losses_saved_floats(b, h, w, patch)
    if nsaved == 0:
        raise UprError(-2, "upr_enh_losses_saved_floats")
    return nsaved


def enhanced_image_losses(enhanced: torch.Tensor, img_low: torch.Tensor, base_target: float = 0.6, patch: int = 16):
    """(exposure, colour, spatial-consistency) losses of losses/loss.py:29-58, :351-368, :404-427 from one read of the two
    images (upr_enh_losses_f32).  [B,3,H,W] f32 CUDA each -> (losses [3], saved statistics for enhanced_image_losses_grad)."""
    enhanced = _cuda(enhanced, "enhanced", shape=(None, 3, None, None))
    img_low = _cuda(img_low, "img_low", shape=enhanced.shape, device=enhanced.device)
    b, _, h, w = enhanced.shape
    losses = torch.empty((3,), dtype=torch.float32, device=enhanced.device)
    saved = torch.empty((_saved_floats(b, h, w, int(patch)),), dtype=torch.float32, device=enhanced.device)
    with _dev(enhanced.device):
        ws = _ws("upr_enh_losses_workspace_bytes", (b,), enhanced.device)
        _run("upr_enh_losses_f32", enhanced.data_ptr(), img_low.data_ptr(), b, h, w, float(base_target), int(patch), losses.data_ptr(),
             saved.data_ptr(), ws.data_ptr(), ws.numel())
    return losses, saved


def enhanced_image_losses_grad(enhanced: torch.Tensor, img_low: torch.Tensor, saved: torch.Tensor, upstream3: torch.Tensor,
                               patch: int = 16) -> torch.Tensor:
    """sum_k upstream3[k] * d loss_k / d enhanced in one pass (upr_enh_losses_grad_f32); upstream3: 3 f32 on the device."""
    enhanced = _cuda(enhanced, "enhanced", shape=(None, 3, None, None))
    img_low = _cuda(img_low, "img_low", shape=enhanced.shape, device=enhanced.device)
    b, _, h, w = enhanced.shape
    saved = _cuda(saved, "saved", shape=(_saved_floats(b, h, w, int(patch)),), device=enhanced.device)
    upstream3 = _cuda(upstream3, "upstream3", shape=(3,), device=enhanced.device)
    grad = torch.empty_like(enhanced)
    with _dev(enhanced.device):
        _run("upr_enh_losses_grad_f32", enhanced.data_ptr(), img_low.data_ptr(), b, h, w, int(patch), saved.data_ptr(),
             upstream3.data_ptr(), grad.data_ptr())
    return grad


def edge_smooth_loss(illu: torch.Tensor, img_low: torch.Tensor, lambda_val: float = 10.0, alpha: float = 1.0, want_grad: bool = True):
    """EdgeAwareSmoothnessLoss.forward (losses/loss.py:136-176) and its gradient w.r.t. illu in three launches
    (upr_edge_smooth_loss_f32).  illu [B,Ci,H,W], img_low [B,Cs,H,W] f32 CUDA -> (loss3 [3] = loss, horizontal, vertical terms;
    d loss / d illu or None)."""
    illu = _cuda(illu, "illu", shape=(None, None, None, None))
    b, ci, h, w = illu.shape
    img_low = _cuda(img_low, "img_low", shape=(b, None, h, w), device=illu.device)
    cs = img_low.shape[1]
    loss3 = torch.empty((3,), dtype=torch.float32, device=illu.device)
    grad = torch.empty_like(illu) if want_grad else None
    with _dev(illu.device):
        ws = _ws("upr_smooth_loss_workspace_bytes", (b, h, w), illu.device)
        _run("upr_edge_smooth_loss_f32", illu.data_ptr(), img_low.data_ptr(), b, ci, cs, h, w, float(lambda_val), float(alpha),
             loss3.data_ptr(), grad.data_ptr() if grad is not None else None, ws.data_ptr(), ws.numel())
    return loss3, grad


def texture_weight_peer(x: torch.Tensor, method: str, weight_smooth: float, peer_table: Optional[torch.Tensor], rank: int,
                        world: int, seq: int):
    """One kernel per rank: per-image texture complexity, the [sum, count] exchange with every peer over NVLink-mapped
    symmetric memory, and the dynamic smoothness weight (upr_texture_weight_peer_f32).
    -> (per_image [B], stats [2] over all ranks, weight 0-dim).  peer_table: int64 CUDA tensor of `world` buffer addresses
    (None = single process)."""
    if method not in ("tv", "edge_density"):
        raise ValueError(f"unsupported texture complexity method: {method}")
    x = _cuda(x, "x")
    if peer_table is not None:
        peer_table = _cuda(peer_table, "peer_table", torch.int64, device=x.device)
        if peer_table.numel() < world:
            raise ValueError(f"peer_table holds {peer_table.numel()} buffer addresses for {world} ranks")
    b, c, h, w = x.shape
    out = torch.empty((b,), dtype=torch.float32, device=x.device)
    stats = torch.empty((2,), dtype=torch.float32, device=x.device)
    weight = torch.empty((), dtype=torch.float32, device=x.device)
    with _dev(x.device):
        ws = _ws("upr_texture_workspace_bytes", (b,), x.device, "tex")
        _run("upr_texture_weight_peer_f32", x.data_ptr(), b, c, h, w, 0 if method == "tv" else 1, out.data_ptr(), stats.data_ptr(),
             ws.data_ptr(), ws.numel(), peer_table.data_ptr() if peer_table is not None else None, int(rank), int(world), int(seq),
             float(weight_smooth), weight.data_ptr())
    return out, stats, weight


def dynamic_smooth_weight(batch_stats2: torch.Tensor, weight_smooth: float = 1.0) -> torch.Tensor:
    """0-dim f32 CUDA tensor: clamp(w0 * (1 - 0.8 * stats[0]/stats[1]), 0.1, 5.0)."""
    s = _cuda(batch_stats2, "batch_stats2", shape=(2,))
    out = torch.empty((), dtype=torch.float32, device=s.device)
    with _dev(s.device):
        _run("upr_dynamic_smooth_weight_f32", s.data_ptr(), float(weight_smooth), out.data_ptr())
    return out


def peer_stats_buffer_bytes() -> int:
    """Bytes of the exchange buffer that every rank gives texture_weight_peer (upr_peer_stats_buffer_bytes)."""
    return lib().upr_peer_stats_buffer_bytes()


def peer_set_timeout_ms(ms: float) -> None:
    """Wall-clock bound on texture_weight_peer's wait for a peer, for every later call in this process (upr_peer_set_timeout_ms)."""
    check(lib().upr_peer_set_timeout_ms(float(ms)), "upr_peer_set_timeout_ms")


def peer_status(buf: torch.Tensor) -> Tuple[int, int]:
    """(sequence number of the exchange that timed out, rank it waited for) from this rank's exchange buffer; (0, 0) = no
    failure so far.  Synchronises the current stream (upr_peer_status)."""
    buf = _cuda(buf, "buf")
    need, have = peer_stats_buffer_bytes(), buf.numel() * buf.element_size()
    if have < need:
        raise ValueError(f"buf must hold the {need} bytes of an exchange buffer, got {have}")
    st = (C.c_uint * 2)()
    with _dev(buf.device):
        _run("upr_peer_status", buf.data_ptr(), st)
    return st[0], st[1]


# ------------------------------------------------------------------------------------------------
# N2: letterbox (utils/letterbox.py) -- geometry by the caller, pixels on the device
# ------------------------------------------------------------------------------------------------
def letterbox(x: torch.Tensor, resized_hw, top: int, left: int, out_hw, pad_value=(114, 114, 114)) -> torch.Tensor:
    """x: [N,C,H,W] f32 CUDA in [0,1]  or  [N,H,W,C] u8 CUDA (decoded files) -> [N,C,oh,ow] f32 CUDA.
    Down-scaling only (bit-exact against cv2.resize INTER_LINEAR on uint8); raises UprError(UPR_E_PARAM) for up-scaling."""
    u8 = isinstance(x, torch.Tensor) and x.dtype == torch.uint8
    x = _cuda(x, "x", torch.uint8 if u8 else torch.float32)
    if u8:
        n, h, w, c = x.shape
    else:
        n, c, h, w = x.shape
    rh, rw = int(resized_hw[0]), int(resized_hw[1])
    oh, ow = int(out_hw[0]), int(out_hw[1])
    out = torch.empty((n, c, oh, ow), dtype=torch.float32, device=x.device)
    pad = (C.c_ubyte * 4)(*([int(v) for v in pad_value] + [114] * 4)[:4])
    with _dev(x.device):
        _run("upr_letterbox_u8_f32" if u8 else "upr_letterbox_f32", x.data_ptr(), out.data_ptr(), n, c, h, w, rh, rw, int(top),
             int(left), oh, ow, pad)
    return out
