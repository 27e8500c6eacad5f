"""Drop-in for the reference's ``enhancers/multi_scale.py`` (same class / method names and return arity).

Reference behaviour mirrored (file:line relative to the reference tree):
  * extract_multi_scale_features   enhancers/multi_scale.py:17-60
  * apply_multi_scale_enhancement  enhancers/multi_scale.py:62-100
  * enhance_with_pyramid           enhancers/multi_scale.py:102-115

Deviations (none changes a numerical result beyond the stated fp32 tolerance):
  * the gain never visits the host: the reference does three ``.item()`` syncs (:90-94), here the
    three means and the gain stay in device memory and feed the clamp kernel directly;
  * batches [N,3,H,W] are accepted, each image gets its own gain (the reference is batch 1).
"""
from __future__ import annotations

import torch

from .. import native
from .adaptive_params import _as_batch, _to_device, cnn_maps


class MultiScaleEnhancer:
    SCALE_WEIGHTS = (0.5, 0.3, 0.2)   # multi_scale.py:87

    def __init__(self):
        pass

    def extract_multi_scale_features(self, image_tensor):
        """List of three [N,7,h_s,w_s] tensors: RGB, luma, per-channel gradient magnitude at scales 1, 1/2, 1/4."""
        x = _to_device(_as_batch(image_tensor))
        f1, f2, f3, _means, _gain = native.multiscale_features(x)
        return [f1, f2, f3]

    def multi_scale_gain(self, image_tensor):
        """(means [N,3], gain [N]) on the device: gain = 1 + 0.1 * sum_s w_s * mean(features_s)."""
        return native.multiscale_stats(_to_device(_as_batch(image_tensor)))

    def apply_multi_scale_enhancement(self, model, image_tensor, device):
        image_tensor = _to_device(_as_batch(image_tensor), device)
        with torch.no_grad():
            maps = cnn_maps(model, image_tensor)
            if maps is not None:
                # the Retinex recombination formed in the gain pass; bit-identical to model(x)[0] -> multiscale_enhance
                illu_map, e_map = maps
                out, _means, _gain = native.retinex_multiscale(image_tensor.contiguous(), illu_map, e_map,
                                                               autocast=torch.is_autocast_enabled("cuda"))
                return out, illu_map
            enhanced_img, _reflectance, illu_map = model(image_tensor)
        # statistics of the input + gain/clamp of the CNN output in one call (chunked on two streams for large batches)
        out, _means, _gain = native.multiscale_enhance(image_tensor, enhanced_img.contiguous())
        return out, illu_map

    def enhance_with_pyramid(self, model, image_tensor, device):
        return self.apply_multi_scale_enhancement(model, image_tensor, device)
