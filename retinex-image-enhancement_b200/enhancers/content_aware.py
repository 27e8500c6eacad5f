"""Drop-in for the reference's ``enhancers/content_aware.py`` (same class / method names and return arity).

Reference behaviour mirrored (file:line relative to the reference tree):
  * compute_saliency_map             enhancers/content_aware.py:19-59
  * compute_attention_map            enhancers/content_aware.py:61-91
  * apply_content_aware_enhancement  enhancers/content_aware.py:93-122

Deviations:
  * the reference computes the saliency on the host and multiplies it with a device tensor
    (content_aware.py:85), which raises on CUDA; here everything is on the device, so the class works
    with ``device='cuda'`` -- the values are the ones the reference produces on CPU;
  * ``compute_saliency_map`` / ``compute_attention_map`` return CPU tensors like the reference unless
    ``keep_on_device=True``; batches are accepted (per-image min/max normalisation).
"""
from __future__ import annotations

import torch

from .. import native
from .adaptive_params import _as_batch, _to_device, cnn_maps


class ContentAwareEnhancer:
    def __init__(self):
        pass

    def compute_saliency_map(self, image_tensor, keep_on_device: bool = False):
        sal = native.saliency(_to_device(_as_batch(image_tensor)))
        return sal if keep_on_device else sal.cpu()

    def compute_attention_map(self, image_tensor, keep_on_device: bool = False):
        att = native.attention(_to_device(_as_batch(image_tensor)))
        return att if keep_on_device else att.cpu()

    def apply_content_aware_enhancement(self, model, image_tensor, device):
        image_tensor = _to_device(_as_batch(image_tensor), device)
        with torch.no_grad():
            maps = cnn_maps(model, image_tensor)
            if maps is not None:
                # the Retinex recombination formed in the attention pass: R and enhanced are never written; bit-identical to
                # model(x)[0] -> content_aware_apply (under the caller's torch.autocast too)
                illu_map, e_map = maps
                return native.retinex_content_aware(image_tensor.contiguous(), illu_map, e_map,
                                                    autocast=torch.is_autocast_enabled("cuda")), illu_map
            enhanced_img, _reflectance, illu_map = model(image_tensor)
        # attention map + gain + clamp in three passes over the frame (the map itself is not materialised)
        return native.content_aware_apply(image_tensor, enhanced_img.contiguous()), illu_map
