"""EXTENSION ops (SURVEY.md section 8f, N4): a generic Gaussian blur, a Gaussian pyramid, log-domain single/multi-scale
Retinex and gamma.  The north-star names them; the reference does NOT contain them (its pyramid is bilinear, it has no
log-domain Retinex and gamma only appears as a training augmentation), so they have no reference parity target and no
reference-facing entry point calls them.  Semantics are OpenCV's / NumPy's (tests compare against cv2 / numpy directly).

All functions take and return float32 CUDA tensors [N,C,H,W]; there is no CPU path.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import torch

from . import native


def _prep(x: torch.Tensor) -> torch.Tensor:
    return native._cuda(x, "x", shape=(None, None, None, None))


def gaussian_blur(x: torch.Tensor, ksize: int, sigma: float = 0.0) -> torch.Tensor:
    """cv2.GaussianBlur(plane, (ksize, ksize), sigma, borderType=cv2.BORDER_REFLECT_101) on every plane (odd ksize <= 31)."""
    x = _prep(x)
    n, c, h, w = x.shape
    out = torch.empty_like(x)
    with native._dev(x.device):
        native._run("upr_ext_gaussian_blur_f32", x.data_ptr(), out.data_ptr(), n * c, h, w, int(ksize), float(sigma))
    return out


def multi_scale_retinex(x: torch.Tensor, ksizes: Sequence[int] = (7, 15, 31), sigmas: Optional[Sequence[float]] = None,
                        weights: Optional[Sequence[float]] = None, eps: float = 1e-6) -> torch.Tensor:
    """sum_s w_s * (log(x + eps) - log(GaussianBlur(x, ksize_s, sigma_s) + eps)); one scale = single-scale Retinex.
    Up to 4 scales, odd ksize <= 31; default weights 1/len(ksizes), default sigmas 0 (= OpenCV's ksize-derived sigma)."""
    x = _prep(x)
    n, c, h, w = x.shape
    k = len(ksizes)
    sigmas = [0.0] * k if sigmas is None else list(sigmas)
    weights = [1.0 / k] * k if weights is None else list(weights)
    if not (len(sigmas) == len(weights) == k):
        raise ValueError("ksizes, sigmas and weights must have the same length")
    out = torch.empty_like(x)
    ks = (C.c_int * k)(*[int(v) for v in ksizes])
    sg = (C.c_double * k)(*[float(v) for v in sigmas])
    wt = (C.c_float * k)(*[float(v) for v in weights])
    with native._dev(x.device):
        native._run("upr_ext_msr_f32", x.data_ptr(), out.data_ptr(), n * c, h, w, k, ks, sg, wt, float(eps))
    return out


def single_scale_retinex(x: torch.Tensor, ksize: int = 15, sigma: float = 0.0, eps: float = 1e-6) -> torch.Tensor:
    return multi_scale_retinex(x, (ksize,), (sigma,), (1.0,), eps)


def pyr_down(x: torch.Tensor) -> torch.Tensor:
    """cv2.pyrDown on every plane: [N,C,H,W] -> [N,C,(H+1)//2,(W+1)//2]."""
    x = _prep(x)
    n, c, h, w = x.shape
    out = torch.empty((n, c, (h + 1) // 2, (w + 1) // 2), dtype=torch.float32, device=x.device)
    with native._dev(x.device):
        native._run("upr_ext_pyr_down_f32", x.data_ptr(), out.data_ptr(), n * c, h, w)
    return out


def gaussian_pyramid(x: torch.Tensor, levels: int = 3) -> List[torch.Tensor]:
    """[x, pyrDown(x), pyrDown(pyrDown(x)), ...] with `levels` entries."""
    pyr = [_prep(x)]
    for _ in range(levels - 1):
        pyr.append(pyr_down(pyr[-1]))
    return pyr


def gamma_correct(x: torch.Tensor, gamma: float) -> torch.Tensor:
    """clamp(x, 0, 1) ** gamma."""
    x = native._cuda(x, "x")
    out = torch.empty_like(x)
    with native._dev(x.device):
        native._run("upr_ext_gamma_f32", x.data_ptr(), out.data_ptr(), x.numel(), float(gamma))
    return out
