"""The oracle against the UNMODIFIED upstream reference, live, on random shapes (CPU; runs where UPR_REFERENCE names a checkout
of xh92117/Retinex-image-Enhancement and is skipped elsewhere).  The golden files pin a handful of fixed inputs; this sweeps
shapes, content kinds and batch rows nobody picked by hand, so that `oracle/` keeps meaning "what the reference computes"
wherever the GPU parity tests use it.

Reference functions executed (paths relative to the reference root): enhancers/adaptive_params.py
AdaptiveParameterAdjuster.{apply_clahe_enhancement, calculate_brightness_features, adjust_parameters}; enhancers/multi_scale.py
MultiScaleEnhancer.extract_multi_scale_features (+ the factor of :87-94); enhancers/content_aware.py
ContentAwareEnhancer.{compute_saliency_map, compute_attention_map}; losses/loss.py calculate_texture_complexity."""
import importlib.util
import os
import sys

import numpy as np
import pytest

REF = os.environ.get("UPR_REFERENCE", "")
pytestmark = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "enhancers")), reason="set UPR_REFERENCE to an unmodified checkout of xh92117/Retinex-image-Enhancement to run this comparison")

torch = pytest.importorskip("torch")
pytest.importorskip("cv2")
from oracle import oracle as O  # noqa: E402

KINDS = ("uniform", "dark", "ramp", "const")


def _load(rel, name):
    """One reference file as an isolated module (no sys.path changes: the reference's package names are generic)."""
    sys.dont_write_bytecode = True
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="module")
def ref():
    ap = _load("enhancers/adaptive_params.py", "_ref_adaptive_params")
    ms = _load("enhancers/multi_scale.py", "_ref_multi_scale")
    ca = _load("enhancers/content_aware.py", "_ref_content_aware")
    return {"adj": ap.AdaptiveParameterAdjuster(), "ms": ms.MultiScaleEnhancer(), "ca": ca.ContentAwareEnhancer()}


def _frame(rng, h, w):
    return O.kat_input(int(rng.integers(1 << 30)), h, w, KINDS[int(rng.integers(len(KINDS)))])


def test_clahe_and_brightness_random_shapes(ref):
    rng = np.random.default_rng(31001)
    for case in range(25):
        h, w = int(rng.integers(8, 260)), int(rng.integers(8, 340))
        x = _frame(rng, h, w)
        want = ref["adj"].apply_clahe_enhancement(torch.from_numpy(x)).contiguous().numpy()
        got = O.clahe_lab(x[0])
        assert np.array_equal(got, want), (case, h, w)
        feats = ref["adj"].calculate_brightness_features(torch.from_numpy(x))
        mine = O.brightness_features(x)
        for k, v in feats.items():
            assert abs(float(mine[k]) - float(v)) <= 1e-12, (case, h, w, k)
        assert O.adjust_parameters(x) == ref["adj"].adjust_parameters(torch.from_numpy(x)), (case, h, w)


def test_multiscale_random_shapes(ref):
    rng = np.random.default_rng(31002)
    for case in range(25):
        h, w = int(rng.integers(4, 200)), int(rng.integers(4, 300))
        x = _frame(rng, h, w)
        feats = ref["ms"].extract_multi_scale_features(torch.from_numpy(x))
        means = [float(torch.mean(f).item()) for f in feats]
        factor = 1.0
        for wt, m in zip([0.5, 0.3, 0.2], means):
            factor += wt * m * 0.1
        m_mine, f_mine = O.multiscale_means(x)
        np.testing.assert_allclose(m_mine, means, rtol=2e-6, atol=1e-7, err_msg=str((case, h, w)))
        assert abs(f_mine - factor) <= 2e-7 * factor, (case, h, w)


def test_saliency_attention_random_shapes(ref):
    rng = np.random.default_rng(31003)
    for case in range(20):
        h, w = int(rng.integers(3, 160)), int(rng.integers(3, 220))
        x = _frame(rng, h, w)
        sal = ref["ca"].compute_saliency_map(torch.from_numpy(x)).numpy()
        att = ref["ca"].compute_attention_map(torch.from_numpy(x)).numpy()
        np.testing.assert_allclose(O.saliency(x), sal, rtol=0, atol=1e-6, err_msg=str((case, h, w)))
        np.testing.assert_allclose(O.attention(x), att, rtol=0, atol=2e-6, err_msg=str((case, h, w)))


def test_texture_complexity_random_shapes():
    # losses/loss.py imports torchvision (for the perceptual loss); the function under test is plain torch
    pytest.importorskip("torchvision")
    loss = _load("losses/loss.py", "_ref_loss")
    rng = np.random.default_rng(31004)
    for case in range(20):
        b, h, w = int(rng.integers(1, 5)), int(rng.integers(3, 120)), int(rng.integers(3, 160))
        x = np.concatenate([_frame(rng, h, w) for _ in range(b)])
        tv = loss.calculate_texture_complexity(torch.from_numpy(x), "tv").numpy()
        ed = loss.calculate_texture_complexity(torch.from_numpy(x), "edge_density").numpy()
        np.testing.assert_allclose(O.texture_tv(x), tv, rtol=2e-6, atol=1e-7, err_msg=str((case, b, h, w)))
        assert np.abs(O.texture_edge_density(x) - ed).max() <= 4.0 / (h * w) + 1e-7, (case, b, h, w)
