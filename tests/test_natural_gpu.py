"""GPU parity on NATURAL image content: crops of the reference's own sample photographs (tests/golden/natural.npz, made by
tests/golden/make_golden_natural.py from the reference's data/input/*.jpg), checked against (i) what the unmodified reference
computed on them (hashes, scalars, sub-sampled maps) and (ii) the oracle's full maps; and the same content mirrored / tiled up to
the BASELINE shapes (1080p, 4K) against the oracle.  Everything goes through the C ABI.

Tolerances: a1 bit-exact; a3 exact histogram, features <= 1e-12; a4/a5 2e-6 relative; a6/a7 2e-6 / 4e-6 absolute on [0,1] maps
(stated bound 1e-4, SURVEY 8c); a9 tv 2e-6 relative, edge density <= 4/N.
"""
import hashlib

import numpy as np
import pytest
import torch

from conftest import mirror_tile, natural_input
from oracle import oracle as O

pytestmark = pytest.mark.gpu


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


@pytest.fixture(scope="module")
def native():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from retinex_image_enhancement_b200 import native as nat
    assert nat.lib().upr_device_check() == 0
    return nat


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def test_natural_crops_match_the_reference(native, natural):
    from retinex_image_enhancement_b200.enhancers.adaptive_params import AdaptiveParameterAdjuster
    meta, arrays = natural
    sub = meta["sub"]
    adj = AdaptiveParameterAdjuster()
    for rec in meta["cases"]:
        name = rec["name"]
        x = natural_input(arrays, name)
        xd = dev(x)
        # a1: bit-exact against the reference's output hash, through the f32 entry, the packed-u8 entry and f32 -> u8
        out = native.clahe_lab(xd).cpu().numpy()
        assert sha(out) == rec["clahe"]["sha_out"], name
        u8 = torch.from_numpy(arrays[f"{name}_u8"][None]).cuda()
        out8 = native.clahe_lab_u8(u8).cpu().numpy()
        assert np.array_equal(out8[0].transpose(2, 0, 1).astype(np.float32) / np.float32(255.0), out[0]), name
        assert np.array_equal(native.clahe_lab_f32_u8(xd).cpu().numpy(), out8), name
        # a3
        f = adj.calculate_brightness_features(torch.from_numpy(x))
        for k, v in rec["bright"]["features"].items():
            assert abs(f[k] - v) <= 1e-12, (name, k)
        assert adj.adjust_parameters(torch.from_numpy(x)) == rec["bright"]["params"]
        # a4 / a5
        means, gain = native.multiscale_stats(xd)
        np.testing.assert_allclose(means.cpu().numpy()[0], rec["multiscale"]["means"], rtol=2e-6)
        assert abs(float(gain[0]) - rec["multiscale"]["factor"]) <= 2e-7 * rec["multiscale"]["factor"] + 6e-8
        # a6 / a7: sub-sampled maps of the reference, full maps of the oracle
        sal, att = native.saliency(xd).cpu().numpy(), native.attention(xd).cpu().numpy()
        np.testing.assert_allclose(sal[0, 0, ::sub, ::sub], arrays[f"{name}_sal_sub"], rtol=0, atol=2e-6)
        np.testing.assert_allclose(att[0, 0, ::sub, ::sub], arrays[f"{name}_att_sub"], rtol=0, atol=4e-6)
        np.testing.assert_allclose(sal, O.saliency(x), rtol=0, atol=2e-6)
        np.testing.assert_allclose(att, O.attention(x), rtol=0, atol=4e-6)
        assert int(sal.argmax()) == rec["content"]["sal_argmax"] and int(att.argmax()) == rec["content"]["att_argmax"]
        # a9
        tv = float(native.texture_complexity(xd, "tv")[0])
        assert abs(tv - rec["texture"]["tv"]) <= 2e-6 * rec["texture"]["tv"]
        ed = float(native.texture_complexity(xd, "edge_density")[0])
        assert abs(ed - rec["texture"]["edge_density"]) <= 4.0 / (rec["h"] * rec["w"])


@pytest.mark.parametrize("h,w", [(1080, 1920), (2160, 3840)])
def test_natural_content_at_baseline_shapes(native, natural, h, w):
    """The photographs mirrored and tiled up to 1080p / 4K (smooth regions, real edges, a near-black border -- nothing like
    noise): every op against the oracle, full frames."""
    _meta, arrays = natural
    names = ["road_stripe", "dark_edge"]
    x = np.concatenate([mirror_tile(natural_input(arrays, nm), h, w) for nm in names])
    enh = np.clip(x * np.float32(1.7) + np.float32(0.05), 0, None).astype(np.float32)
    xd = dev(x)
    out = native.clahe_lab(xd).cpu().numpy()
    means, gain = native.multiscale_stats(xd)
    sal, att = native.saliency(xd).cpu().numpy(), native.attention(xd).cpu().numpy()
    ca = native.content_aware_apply(xd, dev(enh)).cpu().numpy()
    hist = native.brightness_hist(xd).cpu().numpy()
    for i in range(len(names)):
        xi = x[i:i + 1]
        assert np.array_equal(out[i:i + 1], O.clahe_lab(xi)), names[i]
        m_ref, f_ref = O.multiscale_means(xi)
        np.testing.assert_allclose(means.cpu().numpy()[i], m_ref, rtol=2e-6)
        assert abs(float(gain[i]) - f_ref) <= 2e-7 * f_ref + 6e-8
        a_ref = O.attention(xi)
        np.testing.assert_allclose(sal[i:i + 1], O.saliency(xi), rtol=0, atol=2e-6)
        np.testing.assert_allclose(att[i:i + 1], a_ref, rtol=0, atol=4e-6)
        np.testing.assert_allclose(ca[i:i + 1], O.attention_apply(enh[i], a_ref), rtol=0, atol=2e-6)
        assert np.array_equal(hist[i].astype(np.uint32), O.brightness_hist(xi))
