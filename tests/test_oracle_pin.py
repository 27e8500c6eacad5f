"""Pins the CPU oracle (oracle/upr_oracle.c) before anything is allowed to trust it.

Two independent anchors:
  * golden vectors produced by the UNMODIFIED reference (tests/golden/make_golden.py);
  * the cv2 binary itself (the third-party dependency that holds the arithmetic):
    exhaustive 2^24 sweeps for RGB->Lab, Lab->RGB, RGB->Gray and CLAHE on ragged shapes.
"""
import hashlib
import os

import numpy as np
import pytest

from oracle import oracle as O

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

cv2 = pytest.importorskip("cv2")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


@pytest.fixture(scope="module")
def cube():
    r, g, b = np.meshgrid(*(np.arange(256, dtype=np.uint8),) * 3, indexing="ij")
    planar = np.stack([r.ravel(), g.ravel(), b.ravel()])
    hwc = np.ascontiguousarray(planar.T.reshape(4096, 4096, 3))
    return planar, hwc


def test_tables_spot_values():
    t = O.tables()
    assert list(t["gamma"][:6]) == [0, 1, 1, 2, 2, 3] and list(t["gamma"][253:]) == [2004, 2022, 2040]
    # entries where a float64 / libm-cbrtf build would differ (see upr_oracle.c)
    assert t["cbrt"][49] == 9454 and t["cbrt"][628] == 22126 and t["cbrt"][324] == 17745
    assert list(t["y"][:3]) == [0, 7, 14] and t["y"][255] == 16384
    assert t["ify"][0] == 2260 and t["ify"][255] == 16384
    assert list(t["invgamma"][:10]) == [0, 1, 2, 2, 3, 4, 5, 6, 6, 7]


def test_rgb2lab_exhaustive_vs_cv2(cube):
    planar, hwc = cube
    ref = cv2.cvtColor(np.ascontiguousarray(hwc[:, :, ::-1]), cv2.COLOR_BGR2LAB).reshape(-1, 3).T
    assert np.array_equal(O.rgb2lab_u8(planar), ref)


def test_lab2rgb_exhaustive_vs_cv2(cube):
    planar, hwc = cube
    bgr = cv2.cvtColor(hwc, cv2.COLOR_LAB2BGR)
    ref = cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB).reshape(-1, 3).T
    assert np.array_equal(O.lab2rgb_u8(planar), ref)


def test_gray_exhaustive_vs_cv2(cube):
    planar, hwc = cube
    ref = cv2.cvtColor(np.ascontiguousarray(hwc[:, :, ::-1]), cv2.COLOR_BGR2GRAY).ravel()
    assert np.array_equal(O.gray_u8(planar), ref)


def test_quantize_matches_numpy_cast():
    rng = np.random.default_rng(5)
    x = np.concatenate([rng.random(4096, dtype=np.float32) * 3 - 1,
                        np.array([0, 1, 1.5, -0.5, 0.999999, 255 / 255, 254.9999 / 255, np.nan, np.inf, -np.inf,
                                  1e10, -1e10, 8421504.5, -8421504.5, 1e-45, -0.0], np.float32)])
    with np.errstate(invalid="ignore"):
        ref = (x * 255).astype(np.uint8)
    assert np.array_equal(O.quantize_u8(x), ref)


def test_u8_boundary_casts_are_exact():
    """The packed u8 entries (upr_clahe_lab_u8 / upr_clahe_lab_f32_u8) rest on two identities of the reference's own casts:
    the quantiser of adaptive_params.py:142 is the identity on k / 255 (what ToTensor makes of a decoded file), and
    save_image's (y * 255).astype(u8) (enhancers/simple_enhance.py:91-93) recovers k from the op's output k / 255."""
    import torch
    k = np.arange(256, dtype=np.float32)
    assert np.array_equal(O.quantize_u8(k / np.float32(255)), np.arange(256, dtype=np.uint8))
    assert np.array_equal(((k / np.float32(255)) * 255).astype(np.uint8), np.arange(256, dtype=np.uint8))
    t = torch.arange(256, dtype=torch.uint8).float().div(255)      # torchvision ToTensor
    assert np.array_equal(O.quantize_u8(t.numpy()), np.arange(256, dtype=np.uint8))
    # and the reference's cv2 chain on a u8 image equals the oracle on u8 / 255, truncated back
    rng = np.random.default_rng(12)
    img = rng.integers(0, 256, size=(96, 120, 3), dtype=np.uint8)            # RGB, HWC
    bgr = np.ascontiguousarray(img[:, :, ::-1])
    lab = cv2.cvtColor(bgr, cv2.COLOR_BGR2LAB)
    l, a, b = cv2.split(lab)
    l = cv2.createCLAHE(clipLimit=2.0, tileGridSize=(8, 8)).apply(l)
    want = cv2.cvtColor(cv2.merge((l, a, b)), cv2.COLOR_LAB2BGR)[:, :, ::-1]
    xf = np.ascontiguousarray((img.astype(np.float32) / np.float32(255)).transpose(2, 0, 1)[None])
    got = (O.clahe_lab(xf)[0] * np.float32(255)).astype(np.uint8).transpose(1, 2, 0)
    assert np.array_equal(got, want)
    from oracle import cv2_chain
    assert np.array_equal(cv2_chain.clahe_lab_frame_u8(img), want)     # bench.py's CPU arm at the u8 boundary


@pytest.mark.parametrize("shape", [(400, 600), (1080, 1920), (403, 601), (400, 601), (401, 600), (64, 64),
                                   (17, 23), (135, 240), (9, 9)])
@pytest.mark.parametrize("kind", ["uniform", "dark", "const", "ramp"])
def test_clahe_vs_cv2(shape, kind):
    h, w = shape
    rng = np.random.default_rng(h * 131 + w)
    if kind == "uniform":
        src = rng.integers(0, 256, (h, w), dtype=np.uint8)
    elif kind == "dark":
        src = rng.integers(0, 77, (h, w), dtype=np.uint8)
    elif kind == "const":
        src = np.full((h, w), 77, np.uint8)
    else:
        src = ((np.arange(w)[None, :] * 255 // max(w - 1, 1)) * np.ones((h, 1))).astype(np.uint8)
    ref = cv2.createCLAHE(clipLimit=2.0, tileGridSize=(8, 8)).apply(src)
    got, hist, lut = O.clahe_u8(src, taps=True)
    assert np.array_equal(got, ref)
    assert np.array_equal(O.clahe_map_u8(src, lut), got)     # the map step alone, fed the LUTs of the same call
    hp, wp = (h, w) if (h % 8 == 0 and w % 8 == 0) else (h + 8 - h % 8, w + 8 - w % 8)
    assert hist.sum() == hp * wp and (hist.sum(1) == hp * wp // 64).all()


@pytest.mark.parametrize("clip,tiles", [(2.0, (8, 8)), (4.0, (4, 4)), (1.0, (16, 8)), (40.0, (8, 8)), (0.0, (8, 8))])
def test_clahe_other_params_vs_cv2(clip, tiles):
    rng = np.random.default_rng(77)
    src = rng.integers(0, 256, (200, 320), dtype=np.uint8)
    ref = cv2.createCLAHE(clipLimit=clip, tileGridSize=tiles).apply(src)
    got, _, lut = O.clahe_u8(src, clip_limit=clip, tiles=tiles, taps=True)
    assert np.array_equal(got, ref)
    assert np.array_equal(O.clahe_map_u8(src, lut, tiles), got)


def test_golden_clahe(golden, small_cases):
    for rec in golden["clahe"]:
        x = O.kat_input(rec["seed"], rec["h"], rec["w"], rec["kind"])
        assert sha(x) == rec["sha_in"]
        out, taps = O.clahe_lab(x, taps=True)
        assert sha(np.transpose(taps["q"], (1, 2, 0))) == rec["sha_u8_hwc"], rec
        assert sha(out) == rec["sha_out"], rec
        key = f"clahe_{rec['seed']}_out_u8"
        if key in small_cases:
            assert np.array_equal(out[0], small_cases[key].astype(np.float32) / np.float32(255.0))


def test_golden_brightness(golden):
    for rec in golden["bright"]:
        x = O.kat_input(rec["seed"], rec["h"], rec["w"], rec["kind"])
        f = O.brightness_features(x)
        for k, v in rec["features"].items():
            assert abs(f[k] - v) <= 1e-12, (k, f[k], v)
        assert O.adjust_parameters(x) == rec["params"]


def test_golden_multiscale(golden):
    for rec in golden["multiscale"]:
        x = O.kat_input(rec["seed"], rec["h"], rec["w"], rec["kind"])
        means, factor = O.multiscale_means(x)
        np.testing.assert_allclose(means, rec["means"], rtol=2e-6)
        assert abs(factor - rec["factor"]) <= 1e-7


@pytest.mark.parametrize("h,w", [(72, 104), (100, 260), (64, 8), (101, 67), (9, 13), (1081, 1919)])
def test_multiscale_feature_maps(h, w):
    """O.multiscale_features against the reference's own torch formulation on the CPU (multi_scale.py:17-60): bilinear
    F.interpolate to (int(h*s), int(w*s)), luma .299/.587/.114, sqrt(gx^2 + gy^2) of torch.gradient -- at exact scales (h, w
    multiples of 4) and inexact ones.  The maps' fp64 means are multiscale_means (both come from one per-pixel function, so the
    golden pins of the means vouch for the maps too).  Largest difference seen: 1.8e-7 absolute on values in [0, 1], i.e. one
    or two fp32 ulps, from the interpolation and the luma evaluated in another fp32 order (the full-scale image and gradients
    are equal); the magnitude is taken in fp64 from torch's gradients."""
    import torch
    import torch.nn.functional as F
    x = O.kat_input(h * 7 + w, h, w, "uniform")
    maps = O.multiscale_features(x)
    means, _ = O.multiscale_means(x)
    xt = torch.from_numpy(x)
    for k, (s, f) in enumerate(zip((1.0, 0.5, 0.25), maps)):
        size = (int(h * s), int(w * s))
        assert f.shape == (7,) + size
        np.testing.assert_allclose(f.astype(np.float64).mean(), means[k], rtol=1e-12, atol=0)
        img = xt if s == 1.0 else F.interpolate(xt, size=size, mode="bilinear", align_corners=False)
        img = img[0]
        luma = 0.299 * img[0] + 0.587 * img[1] + 0.114 * img[2]
        gx, gy = torch.gradient(img, dim=2)[0].double(), torch.gradient(img, dim=1)[0].double()
        mag = torch.sqrt(gx * gx + gy * gy)
        want = torch.cat([img, luma[None]]).numpy()
        np.testing.assert_allclose(f[:4], want, rtol=0, atol=3e-7, err_msg=f"scale {s}: image / luma")
        np.testing.assert_allclose(f[4:], mag.numpy(), rtol=0, atol=3e-7, err_msg=f"scale {s}: |grad|")
        if s == 1.0:
            assert np.array_equal(f[:3], x[0])


def test_golden_content(golden, small_cases):
    for rec in golden["content"]:
        x = O.kat_input(rec["seed"], rec["h"], rec["w"], rec["kind"])
        sal = O.saliency(x)
        att = O.attention(x)
        assert abs(float(sal.astype(np.float64).mean()) - rec["sal_mean"]) <= 1e-7
        assert abs(float(att.astype(np.float64).mean()) - rec["att_mean"]) <= 1e-7
        assert int(att.argmax()) == rec["att_argmax"] and int(sal.argmax()) == rec["sal_argmax"]
        if f"sal_{rec['seed']}" in small_cases:
            np.testing.assert_allclose(sal[0, 0], small_cases[f"sal_{rec['seed']}"], rtol=0, atol=1e-7)
            np.testing.assert_allclose(att[0, 0], small_cases[f"att_{rec['seed']}"], rtol=0, atol=2e-7)


def test_golden_natural_images(natural):
    """The oracle on crops of the reference's own photographs against what the unmodified reference computed on them."""
    from conftest import natural_input
    meta, arrays = natural
    sub = meta["sub"]
    for rec in meta["cases"]:
        x = natural_input(arrays, rec["name"])
        assert sha(x) == rec["sha_in"]
        out = O.clahe_lab(x)
        assert sha(out) == rec["clahe"]["sha_out"], rec["name"]
        f = O.brightness_features(x)
        for k, v in rec["bright"]["features"].items():
            assert abs(f[k] - v) <= 1e-12, (rec["name"], k)
        assert O.adjust_parameters(x) == rec["bright"]["params"]
        m, fac = O.multiscale_means(x)
        np.testing.assert_allclose(m, rec["multiscale"]["means"], rtol=2e-6)
        assert abs(fac - rec["multiscale"]["factor"]) <= 2e-7
        sal, att = O.saliency(x), O.attention(x)
        np.testing.assert_allclose(sal[0, 0, ::sub, ::sub], arrays[f"{rec['name']}_sal_sub"], rtol=0, atol=2e-7)
        np.testing.assert_allclose(att[0, 0, ::sub, ::sub], arrays[f"{rec['name']}_att_sub"], rtol=0, atol=4e-7)
        assert int(sal.argmax()) == rec["content"]["sal_argmax"] and int(att.argmax()) == rec["content"]["att_argmax"]
        assert abs(float(sal.astype(np.float64).mean()) - rec["content"]["sal_mean"]) <= 1e-7
        assert abs(float(O.texture_tv(x)[0]) - rec["texture"]["tv"]) <= 2e-6 * rec["texture"]["tv"]
        assert abs(float(O.texture_edge_density(x)[0]) - rec["texture"]["edge_density"]) <= 4.0 / (rec["h"] * rec["w"])


def test_golden_retinex(small_cases):
    refl, enh = O.retinex_recombine(small_cases["retinex_x"], small_cases["retinex_illu"], small_cases["retinex_e"])
    assert np.array_equal(refl, small_cases["retinex_refl"])
    np.testing.assert_allclose(enh, small_cases["retinex_enh"], rtol=3e-7, atol=0)


def test_golden_texture(golden):
    for rec in golden["texture"]:
        rng = np.random.default_rng(rec["seed"])
        a = rng.random(tuple(rec["shape"]), dtype=np.float32)
        if rec["kind"] == "dark":
            a = a * np.float32(0.3)
        assert sha(a) == rec["sha_in"]
        tv = O.texture_tv(a)
        np.testing.assert_allclose(tv, rec["tv"], rtol=2e-6)
        ed = O.texture_edge_density(a)
        n = rec["shape"][2] * rec["shape"][3]
        assert np.abs(ed - np.array(rec["edge_density"])).max() <= 4.0 / n
        assert abs(O.dynamic_smooth_weight(tv) - rec["w_tv"]) <= 1e-6


def test_cv2_chain_matches_oracle():
    """bench.py's CPU arm (oracle/cv2_chain.py, the reference's own cv2 call sequence) == the C oracle."""
    from oracle import cv2_chain
    for seed, (h, w), kind in [(2, (400, 600), "dark"), (7, (403, 601), "uniform"), (9, (270, 480), "ramp")]:
        x = O.kat_input(seed, h, w, kind)
        assert np.array_equal(np.ascontiguousarray(cv2_chain.clahe_lab_frame(x[0])), O.clahe_lab(x)[0])
    xs = np.concatenate([O.kat_input(40 + i, 64, 96, "uniform") for i in range(4)])
    for got, x in zip(cv2_chain.clahe_lab_batch(xs, workers=3), xs):
        assert np.array_equal(np.ascontiguousarray(got), O.clahe_lab(x)[0])


# ---- letterbox (SURVEY 8f N2): the fixed-point bilinear recipe against the cv2 binary ---------------------------
@pytest.mark.parametrize("sh,sw,dh,dw", [(480, 640, 240, 320), (1000, 1024, 640, 655), (1080, 1920, 360, 640), (123, 457, 77, 301),
                                          (99, 101, 98, 100), (500, 333, 499, 332), (301, 301, 150, 150), (64, 64, 63, 1), (200, 300, 1, 1),
                                          (1080, 1920, 1078, 1917), (777, 1333, 389, 667), (1024, 1000, 625, 640)])
def test_resize_linear_u8_recipe_matches_cv2_downscale(sh, sw, dh, dw):
    cv2 = pytest.importorskip("cv2")
    from oracle import cv2_chain
    src = np.random.default_rng(sh * 7 + dw).integers(0, 256, (sh, sw, 3), dtype=np.uint8)
    for ipp in (True, False):
        if hasattr(cv2, "ipp"):
            cv2.ipp.setUseIPP(ipp)
        ref = cv2.resize(src, (dw, dh), interpolation=cv2.INTER_LINEAR)
        assert np.array_equal(cv2_chain.resize_linear_u8_fixed(src, dw, dh), ref)
    if hasattr(cv2, "ipp"):
        cv2.ipp.setUseIPP(True)


def test_letterbox_ref_is_the_reference_function():
    """oracle/cv2_chain.letterbox_ref against the unmodified reference's utils/letterbox.py (UPR_REFERENCE)."""
    ref_root = os.environ.get("UPR_REFERENCE", "")
    if not os.path.isdir(os.path.join(ref_root, "utils")):
        pytest.skip("set UPR_REFERENCE to an unmodified checkout of xh92117/Retinex-image-Enhancement to run this comparison")
    pytest.importorskip("cv2")
    import importlib.util
    import torch
    spec = importlib.util.spec_from_file_location("ref_letterbox", os.path.join(ref_root, "utils", "letterbox.py"))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    from oracle import cv2_chain
    x = np.random.default_rng(3).random((3, 300, 517), dtype=np.float32)
    for new_shape, scaleup in ((256, False), (640, False), ((200, 333), True)):
        got, ratio, pad = cv2_chain.letterbox_ref(x, new_shape, auto=True, scaleup=scaleup)
        exp, ratio2, pad2 = ref.letterbox_tensor(torch.from_numpy(x), new_shape=new_shape, auto=True, scaleup=scaleup)
        assert np.array_equal(got, exp.numpy()) and ratio == ratio2 and tuple(pad) == tuple(pad2)


# ---- smoothness term (SURVEY 8f N3) against the unmodified reference ----------------------------------------------
def _smooth_cases():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden_smooth", os.path.join(GOLDEN_DIR, "make_golden_smooth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.smooth_cases


def test_golden_smooth_loss():
    """oracle.edge_smooth_loss == losses/loss.py EdgeAwareSmoothnessLoss + torch autograd (tests/golden/make_golden_smooth.py)."""
    smooth_cases = _smooth_cases()
    gold = np.load(os.path.join(GOLDEN_DIR, "smooth_loss.npz"))
    for name, illu, img, lam, alpha in smooth_cases():
        loss, _lh, _lv, grad = O.edge_smooth_loss(illu, img, lam, alpha)
        assert abs(float(loss) - float(gold[f"{name}_loss"])) <= 2e-6 * abs(float(gold[f"{name}_loss"])), name
        g = gold[f"{name}_grad"]
        assert np.abs(grad - g).max() <= 1e-6 * np.abs(g).max() + 1e-12, name
        assert np.array_equal(grad == 0, g == 0), name      # sign(0) = 0 on plateaus


def test_golden_enhanced_image_losses():
    """oracle.enhanced_image_losses == AdaptiveExposureLoss / ColorLoss / SpatialConsistencyLoss of the unmodified reference
    and torch autograd through them (tests/golden/make_golden_smooth.py)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden_smooth", os.path.join(GOLDEN_DIR, "make_golden_smooth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    gold = np.load(os.path.join(GOLDEN_DIR, "smooth_loss.npz"))
    for name, enh, low in mod.enh_cases():
        losses, grads = O.enhanced_image_losses(enh, low)
        for k, tag in enumerate(("exp", "col", "spa")):
            want, g = float(gold[f"{name}_{tag}_loss"]), gold[f"{name}_{tag}_grad"]
            # the colour term squares differences of nearly equal channel means (|d| ~ 5e-3 of means ~ 0.5): the reference's
            # own fp32 torch.mean rounds those means at 1e-7 relative, i.e. d at ~1e-5 relative -- hence the wider band
            rtol = 2e-4 if tag == "col" else 1e-5
            assert abs(float(losses[k]) - want) <= rtol * abs(want), (name, tag, float(losses[k]), want)
            assert np.abs(grads[k] - g).max() <= rtol * np.abs(g).max() + 1e-12, (name, tag)
