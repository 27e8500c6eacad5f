"""ctypes front-end of ``upr_oracle.c`` (the C restatement of the reference path).

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.

Every function takes/returns numpy arrays and mirrors one reference function:

=====================  =====================================================
oracle function        reference (relative to /root/reference)
=====================  =====================================================
clahe_lab              enhancers/adaptive_params.py:121-169
brightness_features    enhancers/adaptive_params.py:24-68
adjust_parameters      enhancers/adaptive_params.py:70-119
multiscale_means       enhancers/multi_scale.py:17-60, :87-94
multiscale_features    enhancers/multi_scale.py:17-60
scale_clamp            enhancers/multi_scale.py:97-98
saliency               enhancers/content_aware.py:19-59
attention              enhancers/content_aware.py:61-91
attention_apply        enhancers/content_aware.py:119-120
retinex_recombine      models/model.py:405-413, :442
texture_tv             losses/loss.py:536-548
texture_edge_density   losses/loss.py:550-579
dynamic_smooth_weight  losses/loss.py:710-717
=====================  =====================================================
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libupr_oracle.so")
_SRC = os.path.join(_HERE, "upr_oracle.c")
_lib = None


def build(force: bool = False) -> str:
    """Compile upr_oracle.c with the system gcc (same flags as oracle/Makefile)."""
    if not force and os.path.exists(_SO) and os.path.getmtime(_SO) >= os.path.getmtime(_SRC):
        return _SO
    os.makedirs(os.path.dirname(_SO), exist_ok=True)
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    base = [cc, "-O2", "-ffp-contract=off", "-fno-fast-math", "-fvisibility=hidden",
            "-shared", "-fPIC", "-o", _SO, _SRC, "-lm"]
    try:
        subprocess.run(base[:2] + ["-fopenmp"] + base[2:], check=True, capture_output=True)
    except (subprocess.CalledProcessError, FileNotFoundError):
        subprocess.run(base, check=True)  # no libgomp: scalar build
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        _lib.orc_multiscale_means_f32.restype = C.c_double
        _lib.orc_texture_tv_f32.restype = C.c_double
        _lib.orc_texture_edge_density_f32.restype = C.c_double
        _lib.orc_dynamic_smooth_weight.restype = C.c_float
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _chw(img) -> np.ndarray:
    a = np.asarray(img, dtype=np.float32)
    if a.ndim == 4:
        assert a.shape[0] == 1, "oracle works on one image"
        a = a[0]
    assert a.ndim == 3
    return np.ascontiguousarray(a)


def tables():
    g = np.zeros(256, np.uint16); c = np.zeros(3072, np.uint16)
    ify = np.zeros(256, np.uint16); y = np.zeros(256, np.uint16); ig = np.zeros(4096, np.uint8)
    lib().orc_get_tables(_p(g), _p(c), _p(ify), _p(y), _p(ig))
    return {"gamma": g, "cbrt": c, "ify": ify, "y": y, "invgamma": ig}


def quantize_u8(x) -> np.ndarray:
    a = np.ascontiguousarray(x, dtype=np.float32)
    q = np.empty(a.shape, np.uint8)
    lib().orc_quantize_u8(_p(a), _p(q), C.c_int64(a.size))
    return q


def rgb2lab_u8(rgb_planar) -> np.ndarray:
    a = np.ascontiguousarray(rgb_planar, dtype=np.uint8)
    assert a.shape[0] == 3
    out = np.empty_like(a)
    lib().orc_rgb2lab_u8(_p(a), _p(out), C.c_int64(a[0].size))
    return out


def lab2rgb_u8(lab_planar) -> np.ndarray:
    a = np.ascontiguousarray(lab_planar, dtype=np.uint8)
    assert a.shape[0] == 3
    out = np.empty_like(a)
    lib().orc_lab2rgb_u8(_p(a), _p(out), C.c_int64(a[0].size))
    return out


def gray_u8(rgb_planar) -> np.ndarray:
    a = np.ascontiguousarray(rgb_planar, dtype=np.uint8)
    out = np.empty(a.shape[1:], np.uint8)
    lib().orc_gray_u8(_p(a), _p(out), C.c_int64(a[0].size))
    return out


def clahe_u8(src, clip_limit=2.0, tiles=(8, 8), taps=False):
    a = np.ascontiguousarray(src, dtype=np.uint8)
    h, w = a.shape
    tx, ty = tiles
    dst = np.empty_like(a)
    hist = np.zeros((ty * tx, 256), np.int32)
    lut = np.zeros((ty * tx, 256), np.uint8)
    rc = lib().orc_clahe_u8(_p(a), _p(dst), h, w, C.c_double(clip_limit), tx, ty, _p(hist), _p(lut))
    if rc:
        raise ValueError(f"orc_clahe_u8 rc={rc}")
    return (dst, hist, lut) if taps else dst


def clahe_map_u8(src, lut, tiles=(8, 8)) -> np.ndarray:
    """The interpolation step of clahe_u8 alone: src [H,W] u8 through the tile LUTs lut [ty*tx,256] u8 -> [H,W] u8."""
    a = np.ascontiguousarray(src, dtype=np.uint8)
    h, w = a.shape
    tx, ty = tiles
    t = np.ascontiguousarray(lut, dtype=np.uint8)
    assert t.shape == (ty * tx, 256), t.shape
    dst = np.empty_like(a)
    rc = lib().orc_clahe_map_u8(_p(a), _p(dst), h, w, tx, ty, _p(t))
    if rc:
        raise ValueError(f"orc_clahe_map_u8 rc={rc}")
    return dst


def clahe_lab(img, clip_limit=2.0, tiles=(8, 8), taps=False):
    """a1.  img: [1,3,H,W] or [3,H,W] f32 -> [1,3,H,W] f32 (C-contiguous)."""
    a = _chw(img)
    _, h, w = a.shape
    tx, ty = tiles
    out = np.empty_like(a)
    q = np.empty((3, h, w), np.uint8); lab = np.empty((3, h, w), np.uint8)
    hist = np.zeros((ty * tx, 256), np.int32); lut = np.zeros((ty * tx, 256), np.uint8)
    rc = lib().orc_clahe_lab_f32(_p(a), _p(out), h, w, C.c_double(clip_limit), tx, ty,
                                 _p(q), _p(lab), _p(hist), _p(lut))
    if rc:
        raise ValueError(f"orc_clahe_lab_f32 rc={rc}")
    out = out[None]
    if taps:
        return out, {"q": q, "lab": lab, "hist": hist, "lut": lut}
    return out


def brightness_hist(img) -> np.ndarray:
    a = _chw(img)
    hist = np.zeros(256, np.uint32)
    lib().orc_brightness_hist_f32(_p(a), a.shape[1], a.shape[2], _p(hist))
    return hist


def features_from_hist(hist) -> dict:
    """adaptive_params.py:52-66 expressed on the 256-bin gray histogram (exact)."""
    h = np.asarray(hist, dtype=np.int64)
    n = int(h.sum())
    k = np.arange(256, dtype=np.float64)
    mean = float((h * k).sum()) / n
    var = float((h * (k - mean) ** 2).sum()) / n
    return {
        "mean_brightness": mean / 255.0,
        "brightness_std": float(np.sqrt(var)) / 255.0,
        "dark_pixel_ratio": float(h[:50].sum()) / n,
        "mid_pixel_ratio": float(h[50:201].sum()) / n,
        "bright_pixel_ratio": float(h[201:].sum()) / n,
    }


def brightness_features(img) -> dict:
    return features_from_hist(brightness_hist(img))


def adjust_parameters(img) -> dict:
    """adaptive_params.py:84-117 threshold rules."""
    f = brightness_features(img)
    p = {"enhance_strength": 1.0, "color_balance": 1.0, "brightness_boost": 1.0, "contrast_adjust": 1.0}
    m, s, d = f["mean_brightness"], f["brightness_std"], f["dark_pixel_ratio"]
    if m < 0.2:
        p["enhance_strength"], p["brightness_boost"] = 1.5, 1.3
    elif m < 0.4:
        p["enhance_strength"], p["brightness_boost"] = 1.3, 1.2
    elif m > 0.7:
        p["enhance_strength"], p["brightness_boost"] = 0.8, 0.9
    p["contrast_adjust"] = 1.3 if s < 0.1 else (1.1 if s < 0.2 else 0.9)
    p["color_balance"] = 1.2 if d > 0.6 else (1.1 if d > 0.3 else 1.0)
    return p


def multiscale_means(img):
    a = _chw(img)
    m = np.zeros(3, np.float64)
    f = lib().orc_multiscale_means_f32(_p(a), a.shape[1], a.shape[2], _p(m))
    return m, float(f)


def multiscale_features(img):
    """a4 feature maps of one image: ([7,H,W], [7,int(H/2),int(W/2)], [7,int(H/4),int(W/4)]) f32, channels
    {R, G, B, luma, |grad R|, |grad G|, |grad B|} -- the values whose means multiscale_means returns."""
    a = _chw(img)
    _, h, w = a.shape
    f = [np.empty((7, int(h * s), int(w * s)), np.float32) for s in (1.0, 0.5, 0.25)]
    if min(f[2].shape[1:]) < 1:
        raise ValueError("image too small for the 1/4 scale")
    rc = lib().orc_multiscale_features_f32(_p(a), h, w, _p(f[0]), _p(f[1]), _p(f[2]))
    if rc:
        raise ValueError(f"orc_multiscale_features_f32 rc={rc}")
    return tuple(f)


def scale_clamp(enh, gain: float) -> np.ndarray:
    a = np.ascontiguousarray(enh, dtype=np.float32)
    out = np.empty_like(a)
    lib().orc_scale_clamp_f32(_p(a), C.c_float(gain), _p(out), C.c_int64(a.size))
    return out


def saliency(img, want_minmax=False):
    a = _chw(img)
    _, h, w = a.shape
    sal = np.empty((h, w), np.float32)
    mm = np.zeros(2, np.float64)
    rc = lib().orc_saliency_f32(_p(a), h, w, _p(sal), _p(mm))
    if rc:
        raise ValueError(f"orc_saliency_f32 rc={rc}")
    sal = sal[None, None]
    return (sal, mm) if want_minmax else sal


def attention(img) -> np.ndarray:
    a = _chw(img)
    _, h, w = a.shape
    att = np.empty((h, w), np.float32)
    rc = lib().orc_attention_f32(_p(a), h, w, _p(att))
    if rc:
        raise ValueError(f"orc_attention_f32 rc={rc}")
    return att[None, None]


def attention_apply(enh, att) -> np.ndarray:
    e = _chw(enh)
    t = np.ascontiguousarray(np.asarray(att, np.float32).reshape(e.shape[1], e.shape[2]))
    out = np.empty_like(e)
    lib().orc_attention_apply_f32(_p(e), _p(t), _p(out), e.shape[1], e.shape[2])
    return out[None]


def retinex_recombine(x, illu, e, eps=1e-6):
    """x,e: [B,3,H,W]; illu: [B,1,H,W] -> (reflectance, enhanced)."""
    x = np.ascontiguousarray(x, np.float32); e = np.ascontiguousarray(e, np.float32)
    illu = np.ascontiguousarray(illu, np.float32)
    refl = np.empty_like(x); enh = np.empty_like(x)
    n = x.shape[2] * x.shape[3]
    for b in range(x.shape[0]):
        lib().orc_retinex_recombine_f32(_p(x[b]), _p(illu[b]), _p(e[b]), _p(refl[b]), _p(enh[b]),
                                        C.c_int64(n), C.c_float(eps))
    return refl, enh


def texture_tv(img) -> np.ndarray:
    a = np.ascontiguousarray(img, np.float32)
    b, c, h, w = a.shape
    return np.array([lib().orc_texture_tv_f32(_p(a[i]), c, h, w) for i in range(b)], np.float32)


def texture_edge_density(img, want_mean=False):
    a = np.ascontiguousarray(img, np.float32)
    b, c, h, w = a.shape
    out = np.zeros(b, np.float32); means = np.zeros(b, np.float64)
    for i in range(b):
        m = C.c_double(0.0)
        out[i] = lib().orc_texture_edge_density_f32(_p(a[i]), c, h, w, C.byref(m))
        means[i] = m.value
    return (out, means) if want_mean else out


def dynamic_smooth_weight(complexity, weight_smooth=1.0) -> float:
    c = np.ascontiguousarray(complexity, np.float32)
    return float(lib().orc_dynamic_smooth_weight(_p(c), int(c.size), C.c_float(weight_smooth)))


def edge_smooth_loss(illu, img_low, lambda_val=10.0, alpha=1.0):
    """EdgeAwareSmoothnessLoss.forward (losses/loss.py:136-176) and d loss / d illu, restated in NumPy (fp32 element-wise like
    the reference, fp64 sums).  illu [B,Ci,H,W], img_low [B,Cs,H,W] -> (loss, loss_h, loss_v, grad [B,Ci,H,W])."""
    I = np.ascontiguousarray(illu, np.float32)
    S = np.ascontiguousarray(img_low, np.float32)
    b, ci, h, w = I.shape
    f32 = np.float32
    # edge map (:110-136): channel mean, reflect pad 1, Sobel cross-correlation, magnitude
    gray = S.mean(axis=1, dtype=np.float32, keepdims=True) if S.shape[1] > 1 else S
    p = np.pad(gray, ((0, 0), (0, 0), (1, 1), (1, 1)), mode="reflect")
    gx = (p[..., :-2, 2:] - p[..., :-2, :-2]) + f32(2) * (p[..., 1:-1, 2:] - p[..., 1:-1, :-2]) + (p[..., 2:, 2:] - p[..., 2:, :-2])
    gy = (p[..., 2:, :-2] - p[..., :-2, :-2]) + f32(2) * (p[..., 2:, 1:-1] - p[..., :-2, 1:-1]) + (p[..., 2:, 2:] - p[..., :-2, 2:])
    edge = np.sqrt(gx * gx + gy * gy).astype(np.float32)                                       # [B,1,H,W]
    # avg_pool2d((1, W-1), stride 1)[..., :-1] is the mean of the first W-1 columns; likewise for rows (:163-164)
    fh = (f32(1) + f32(alpha) * edge[..., : w - 1].mean(axis=3, dtype=np.float64, keepdims=True).astype(np.float32))   # [B,1,H,1]
    fv = (f32(1) + f32(alpha) * edge[..., : h - 1, :].mean(axis=2, dtype=np.float64, keepdims=True).astype(np.float32))  # [B,1,1,W]
    wh = np.exp(f32(-lambda_val) * np.abs(S[..., :-1] - S[..., 1:]).mean(axis=1, dtype=np.float32, keepdims=True)).astype(np.float32)
    wv = np.exp(f32(-lambda_val) * np.abs(S[..., :-1, :] - S[..., 1:, :]).mean(axis=1, dtype=np.float32, keepdims=True)).astype(np.float32)
    dh = I[..., :-1] - I[..., 1:]
    dv = I[..., :-1, :] - I[..., 1:, :]
    ch = (wh * fh).astype(np.float32)          # [B,1,H,W-1]
    cv = (wv * fv).astype(np.float32)          # [B,1,H-1,W]
    loss_h = f32((ch * np.abs(dh)).sum(dtype=np.float64) / dh.size)
    loss_v = f32((cv * np.abs(dv)).sum(dtype=np.float64) / dv.size)
    grad = np.zeros_like(I)
    gh_ = (ch * np.sign(dh)).astype(np.float32) * f32(1.0 / dh.size)
    gv_ = (cv * np.sign(dv)).astype(np.float32) * f32(1.0 / dv.size)
    grad[..., :-1] += gh_
    grad[..., 1:] -= gh_
    grad[..., :-1, :] += gv_
    grad[..., 1:, :] -= gv_
    return f32(loss_h + loss_v), loss_h, loss_v, grad


def enhanced_image_losses(enhanced, img_low, base_target=0.6, patch=16):
    """AdaptiveExposureLoss (losses/loss.py:29-58), ColorLoss (:351-368), SpatialConsistencyLoss (:404-427) and their gradients
    w.r.t. the enhanced image, restated in NumPy.  [B,3,H,W] each -> ((exp, col, spa), (g_exp, g_col, g_spa))."""
    R = np.ascontiguousarray(enhanced, np.float32)
    S = np.ascontiguousarray(img_low, np.float32)
    b, c, h, w = R.shape
    f32 = np.float32
    # exposure
    gray_r = R.mean(axis=1, dtype=np.float32)                                     # [B,H,W]
    gmean = f32(S.mean(axis=1, dtype=np.float32).mean(dtype=np.float64))
    target = f32(base_target) + f32(0.8 - base_target) * (f32(1) - gmean)
    hp, wp = h // patch, w // patch
    pm = gray_r[:, : hp * patch, : wp * patch].reshape(b, hp, patch, wp, patch).mean(axis=(2, 4), dtype=np.float64).astype(np.float32)
    l_exp = f32(np.abs(pm - target).mean(dtype=np.float64))
    g_exp = np.zeros_like(R)
    sg = (np.sign(pm - target) * f32(1.0 / (pm.size * patch * patch * c))).astype(np.float32)
    g_exp[:, :, : hp * patch, : wp * patch] = np.repeat(np.repeat(sg, patch, axis=1), patch, axis=2)[:, None]
    # colour
    m = R.mean(axis=(0, 2, 3), dtype=np.float64).astype(np.float32)
    drg, drb, dgb = m[0] - m[1], m[0] - m[2], m[1] - m[2]
    l_col = f32(drg * drg + drb * drb + dgb * dgb)
    g_col = np.zeros_like(R)
    npix = f32(1.0 / (b * h * w))
    g_col[:, 0] = f32(2) * (drg + drb) * npix
    g_col[:, 1] = f32(2) * (dgb - drg) * npix
    g_col[:, 2] = f32(-2) * (drb + dgb) * npix
    # spatial consistency
    dh = (R[..., :-1] - R[..., 1:]) - (S[..., :-1] - S[..., 1:])
    dv = (R[..., :-1, :] - R[..., 1:, :]) - (S[..., :-1, :] - S[..., 1:, :])
    l_spa = f32(f32((dh * dh).mean(dtype=np.float64)) + f32((dv * dv).mean(dtype=np.float64)))
    g_spa = np.zeros_like(R)
    gh_ = dh * f32(2.0 / dh.size)
    gv_ = dv * f32(2.0 / dv.size)
    g_spa[..., :-1] += gh_
    g_spa[..., 1:] -= gh_
    g_spa[..., :-1, :] += gv_
    g_spa[..., 1:, :] -= gv_
    return (l_exp, l_col, l_spa), (g_exp, g_col, g_spa)


# --------------------------------------------------------------------------- #
# Deterministic KAT inputs (SURVEY.md section 8c)
# --------------------------------------------------------------------------- #
def kat_input(seed: int, h: int, w: int, kind: str) -> np.ndarray:
    rng = np.random.default_rng(seed)
    if kind == "uniform":
        return rng.random((1, 3, h, w), dtype=np.float32)
    if kind == "dark":
        return rng.random((1, 3, h, w), dtype=np.float32) * np.float32(0.3)
    if kind == "ramp":
        x = np.arange(w, dtype=np.float32)[None, :]
        y = np.arange(h, dtype=np.float32)[:, None]
        r = np.broadcast_to(x / np.float32(w - 1), (h, w))
        g = np.broadcast_to(y / np.float32(h - 1), (h, w))
        b = (x + y) / np.float32(h + w - 2)
        return np.ascontiguousarray(np.stack([r, g, b])[None].astype(np.float32))
    if kind == "const":
        return np.full((1, 3, h, w), 0.3, np.float32)
    raise ValueError(kind)
