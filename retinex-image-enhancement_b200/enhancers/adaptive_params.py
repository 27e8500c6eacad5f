"""Drop-in for the reference's ``enhancers/adaptive_params.py`` (same class / method names,
argument meaning and return arity), with the arithmetic done on the B200.

Reference behaviour mirrored (file:line relative to the reference tree):
  * calculate_brightness_features  enhancers/adaptive_params.py:24-68
  * adjust_parameters              enhancers/adaptive_params.py:70-119
  * apply_clahe_enhancement        enhancers/adaptive_params.py:121-169
  * apply_adaptive_enhancement     enhancers/adaptive_params.py:171-200

Documented deviations (none changes a numerical result):
  * inputs may be batches [N,3,H,W]; the reference only works for N == 1;
  * ``apply_clahe_enhancement`` returns a contiguous tensor (the reference returns a permuted
    HWC view with the same values) and accepts ``keep_on_device=True`` to skip the D2H copy;
  * ``apply_adaptive_enhancement`` keeps everything on the device (the reference crosses PCIe
    three times per image, adaptive_params.py:188/:136/:198);
  * the parameter dict the reference computes inside ``apply_adaptive_enhancement`` and never uses
    (adaptive_params.py:185) is formed lazily: the histogram kernel is launched asynchronously on the
    input, the 1 KB D2H copy and the rules run only if ``last_parameters()`` is called -- the enhance
    call itself never synchronises with the host.
"""
from __future__ import annotations

import torch

from .. import native


def _as_batch(image_tensor: torch.Tensor) -> torch.Tensor:
    if image_tensor.dim() == 3:
        image_tensor = image_tensor.unsqueeze(0)
    if image_tensor.dim() != 4 or image_tensor.shape[1] != 3:
        raise ValueError(f"expected [N,3,H,W] or [3,H,W], got {tuple(image_tensor.shape)}")
    return image_tensor


def _to_device(image_tensor: torch.Tensor, device=None) -> torch.Tensor:
    """f32 CUDA copy of ``image_tensor`` (async when the source is pinned)."""
    if image_tensor.is_cuda and device is None:
        return image_tensor.detach().to(torch.float32)
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    return image_tensor.detach().to(device=dev, dtype=torch.float32, non_blocking=True)


def cnn_maps(model, image_tensor: torch.Tensor):
    """(illu, e) = model.forward_maps(x) for the inference modes that take the CNN maps straight into their last pass: a model
    with forward_maps that is not training, a CUDA input, and maps the native *_typed entries accept.  None otherwise, and the
    caller runs model(x) as before (for maps in a pair those entries do not take, that is a second forward pass)."""
    if not (image_tensor.is_cuda and hasattr(model, "forward_maps") and not getattr(model, "training", False)):
        return None
    illu, e = model.forward_maps(image_tensor)
    return (illu.contiguous(), e.contiguous()) if native.maps_supported(image_tensor, illu, e) else None


class AdaptiveParameterAdjuster:
    """Image-statistics driven parameter selection plus the CLAHE-in-Lab post-enhancer."""

    CLIP_LIMIT = 2.0          # adaptive_params.py:149
    TILE_GRID = (8, 8)        # adaptive_params.py:149

    def __init__(self):
        self.default_params = {
            "enhance_strength": 1.0,
            "color_balance": 1.0,
            "brightness_boost": 1.0,
            "contrast_adjust": 1.0,
        }
        self._pending_hist = None

    # -- a3 ------------------------------------------------------------------------------------
    def calculate_brightness_features(self, image_tensor):
        from . import _stats
        hist = _stats.brightness_histogram(_to_device(_as_batch(image_tensor)))
        feats = _stats.features_from_histogram(hist)
        return feats[0] if len(feats) == 1 else feats

    def adjust_parameters(self, image_tensor):
        feats = self.calculate_brightness_features(image_tensor)
        if isinstance(feats, dict):
            return self._rules(feats)
        return [self._rules(f) for f in feats]

    def _rules(self, feats):
        params = dict(self.default_params)
        mean, std, dark = feats["mean_brightness"], feats["brightness_std"], feats["dark_pixel_ratio"]
        if mean < 0.2:
            params.update(enhance_strength=1.5, brightness_boost=1.3)
        elif mean < 0.4:
            params.update(enhance_strength=1.3, brightness_boost=1.2)
        elif mean > 0.7:
            params.update(enhance_strength=0.8, brightness_boost=0.9)
        else:
            params.update(enhance_strength=1.0, brightness_boost=1.0)
        params["contrast_adjust"] = 1.3 if std < 0.1 else (1.1 if std < 0.2 else 0.9)
        params["color_balance"] = 1.2 if dark > 0.6 else (1.1 if dark > 0.3 else 1.0)
        return params

    def note_input(self, image_tensor):
        """What apply_adaptive_enhancement does with its input before the CNN (adaptive_params.py:185), without the host
        round trip: the gray histogram is computed on the device, asynchronously; see ``last_parameters``."""
        self._pending_hist = native.brightness_hist(image_tensor)

    def last_parameters(self):
        """The parameter dict(s) of the most recent apply_adaptive_enhancement input (this call copies 1 KB per image to the
        host and therefore synchronises); None before the first call."""
        if self._pending_hist is None:
            return None
        from . import _stats
        import numpy as np
        feats = _stats.features_from_histogram(self._pending_hist.cpu().numpy().astype(np.int64))
        rules = [self._rules(f) for f in feats]
        return rules[0] if len(rules) == 1 else rules

    # -- a1 ------------------------------------------------------------------------------------
    def apply_clahe_enhancement(self, image_tensor, keep_on_device: bool = False):
        image_tensor = _as_batch(image_tensor)
        if not image_tensor.is_cuda and not keep_on_device:
            # host in -> host out, like the reference (:136 / :164): H2D, kernels and D2H are pipelined
            # inside the library (upr_clahe_lab_f32_host)
            return native.clahe_lab_host(image_tensor.detach().to(torch.float32), self.CLIP_LIMIT, self.TILE_GRID)
        out = native.clahe_lab(_to_device(image_tensor), self.CLIP_LIMIT, self.TILE_GRID)
        return out if keep_on_device else out.cpu()

    # -- a2 ------------------------------------------------------------------------------------
    def apply_adaptive_enhancement(self, model, image_tensor, device):
        # The reference computes the parameter dict here and never uses it (adaptive_params.py:185): the histogram kernel is
        # launched (asynchronously), the dict is available from last_parameters() on demand.
        image_tensor = _to_device(_as_batch(image_tensor), device)
        self.note_input(image_tensor)
        with torch.no_grad():
            if hasattr(model, "forward_maps") and not getattr(model, "training", False):
                # recombination (models/model.py:405-413,442) fused into the CLAHE histogram kernel: the `enhanced` frame
                # is never materialised; bit-identical to model(x)[0] -> apply_clahe_enhancement
                illu_map, e_map = model.forward_maps(image_tensor)
                # (maps from a CNN under the caller's torch.autocast: fp16 / bf16 e, with e**2 evaluated as autocast does)
                enhanced_img = native.retinex_clahe(image_tensor.contiguous(), illu_map.contiguous(), e_map.contiguous(),
                                                    self.CLIP_LIMIT, self.TILE_GRID, autocast=torch.is_autocast_enabled("cuda"))
                return enhanced_img, illu_map
            enhanced_img, _reflectance, illu_map = model(image_tensor)
        enhanced_img = native.clahe_lab(enhanced_img, self.CLIP_LIMIT, self.TILE_GRID)
        return enhanced_img, illu_map
