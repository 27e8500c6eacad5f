"""Inference with the CNN under CUDA autocast: fp16 / bf16 Retinex maps through the fused Retinex + CLAHE kernels
(upr_retinex_clahe_typed_f32 / _u8), the forward recombination (upr_retinex_recombine_typed) and the enhance / predict drivers.

Every result is compared bit for bit with the stock composition on the same operands: the two Retinex lines of
models/model.py:412, :442 in torch eager under torch.autocast("cuda", dtype=e.dtype, enabled=autocast), then clahe_lab /
clahe_lab_f32_u8.  The map pairs are those the entries take: e fp16 / bf16, illu f32 (what the real network emits under
autocast) or e's dtype."""
import os
import random

import numpy as np
import pytest
import torch

EPS = 1e-6
HALVES = (torch.float16, torch.bfloat16)
COMBOS = [(di, de, ac) for de in HALVES for di in (torch.float32, de) for ac in (False, True)]
COMBO_IDS = [f"{str(di)[6:]}-{str(de)[6:]}-{'ac' if ac else 'noac'}" for di, de, ac in COMBOS]
gpu = pytest.mark.gpu


def _lib():
    import __graft_entry__ as g
    g.ensure_built()
    from retinex_image_enhancement_b200 import native
    return native.lib()


# ---- CPU: status codes of the C entries (every pointer NULL, so no order of the checks can reach a launch) -------------------
F32, F16, BF16, AC = 0, 1, 2, 1


def _clahe_call(entry, illu_dt, e_dt, flags, n=1, h=8, w=8, tiles=(2, 2)):
    return entry(None, None, illu_dt, None, e_dt, flags, None, n, h, w, EPS, 2.0, tiles[0], tiles[1], None, 0, None)


def _recombine_call(entry, illu_dt, e_dt, flags, n=1, h=8, w=8):
    return entry(None, None, illu_dt, None, e_dt, flags, None, None, n, h, w, EPS, None)


@pytest.mark.parametrize("name", ["upr_retinex_clahe_typed_f32", "upr_retinex_clahe_typed_u8", "upr_retinex_recombine_typed"])
def test_typed_entries_check_their_arguments(name):
    entry = getattr(_lib(), name)
    call = _recombine_call if name == "upr_retinex_recombine_typed" else _clahe_call
    for illu_dt, e_dt in ((F32, F16), (F32, BF16), (F16, F16), (BF16, BF16), (F32, F32)):
        for flags in (0, AC):
            assert call(entry, illu_dt, e_dt, flags) == -1                    # NULL
            assert call(entry, illu_dt, e_dt, flags, n=0) == 0                # empty batch
    assert call(entry, F32, 3, 0) == -4                                      # unknown e dtype
    assert call(entry, 5, F16, 0) == -4                                      # unknown illu dtype
    assert call(entry, F32, -1, 0) == -4
    assert call(entry, F16, BF16, 0) == -4                                   # illu neither f32 nor e's dtype
    assert call(entry, BF16, F16, AC) == -4
    assert call(entry, F16, F32, 0) == -4
    assert call(entry, F32, F16, 2) == -4                                    # unknown flag
    assert call(entry, F32, F16, AC | 4) == -4
    assert call(entry, F32, F16, 0, h=0) == -2                               # bad shape, checked first
    assert call(entry, F32, F16, 0, n=-1) == -2
    assert call(entry, F16, BF16, 2, w=0) == -2
    assert call(entry, F16, BF16, 0, n=0) == -4                              # dtypes before the empty-batch rule
    if call is _clahe_call:
        assert call(entry, F32, F16, 0, tiles=(0, 2)) == -2
        assert call(entry, F32, F16, 0, tiles=(2, 257)) == -2


def test_amp_option_is_parsed_and_checked():
    from retinex_image_enhancement_b200 import cli
    from retinex_image_enhancement_b200.enhancers.simple_enhance import amp_context
    assert cli.build_main_parser().parse_args(["--amp", "bf16"]).amp == "bf16"
    assert cli.build_main_parser().parse_args([]).amp is None
    with pytest.raises(SystemExit):
        cli.build_main_parser().parse_args(["--amp", "fp8"])
    with pytest.raises(ValueError):
        amp_context("half")
    with amp_context(None):
        assert not torch.is_autocast_enabled("cuda")


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def native():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from retinex_image_enhancement_b200 import native as nat
    assert nat.lib().upr_device_check() == 0
    return nat


def exact(got, want):
    assert got.dtype == want.dtype and got.shape == want.shape
    torch.testing.assert_close(got, want, rtol=0, atol=0, equal_nan=True)


def stock_lines(x, illu, e, autocast):
    """(R, enhanced) of models/model.py:412, :442 in torch eager under CUDA autocast in e's dtype."""
    with torch.autocast("cuda", dtype=e.dtype if e is not None else torch.float16, enabled=autocast):
        r = x / (illu + EPS)
        return r, (None if e is None else r * e + (1 - r) * (e ** 2))


def stock(native, x, illu, e, autocast, u8, tiles=(8, 8)):
    enh = stock_lines(x, illu, e, autocast)[1]
    assert enh.dtype == torch.float32
    return native.clahe_lab_f32_u8(enh, 2.0, tiles) if u8 else native.clahe_lab(enh, 2.0, tiles)


def fused(native, x, illu, e, autocast, u8, tiles=(8, 8), out=None):
    fn = native.retinex_clahe_u8 if u8 else native.retinex_clahe
    return fn(x, illu, e, 2.0, tiles, EPS, out=out, autocast=autocast)


def maps(n, h, w, di, de, seed, misalign=""):
    """x [n,3,h,w] f32 in [0,1), illu in [0.05, 0.95) and e in [0, 1.2) on the GPU; `misalign` names the tensors that start one
    element past an aligned address."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.rand((n, 3, h, w), generator=g)
    illu = (torch.rand((n, 1, h, w), generator=g) * 0.9 + 0.05).to(di)
    e = (torch.rand((n, 3, h, w), generator=g) * 1.2).to(de)
    out = []
    for name, t in (("x", x), ("illu", illu), ("e", e)):
        t = t.cuda()
        if name in misalign:
            buf = torch.empty(t.numel() + 1, dtype=t.dtype, device="cuda")
            t = buf[1:].view(t.shape).copy_(t)
        out.append(t)
    return out


@gpu
def test_real_network_emits_f32_illumination_and_autocast_enhancement_map(native):
    from retinex_image_enhancement_b200.models.model import UP_Retinex
    torch.manual_seed(0)
    model = UP_Retinex(use_preact=False, use_aspp=False).cuda().eval()
    x = torch.rand((1, 3, 64, 96), device="cuda")
    for dt in HALVES:
        with torch.no_grad(), torch.autocast("cuda", dtype=dt):
            illu, e = model.forward_maps(x)
        assert (illu.dtype, e.dtype) == (torch.float32, dt)


SHAPES = [  # (n, h, w, tiles): vector path (1080p, 4K, a batch), then the generic one (padded tiles, grids 2x2 and 16x16)
    (1, 1080, 1920, (8, 8)), (1, 2160, 3840, (8, 8)), (5, 256, 384, (8, 8)),
    (2, 403, 601, (8, 8)), (1, 403, 601, (2, 2)), (1, 403, 601, (16, 16)), (2, 96, 128, (3, 5)),
]


@gpu
@pytest.mark.parametrize("u8", [False, True], ids=["f32", "u8"])
@pytest.mark.parametrize("shape", SHAPES, ids=[f"{n}x{h}x{w}-{t[0]}x{t[1]}" for n, h, w, t in SHAPES])
@pytest.mark.parametrize("combo", COMBOS, ids=COMBO_IDS)
def test_fused_equals_stock_composition(native, combo, shape, u8):
    di, de, ac = combo
    n, h, w, tiles = shape
    x, illu, e = maps(n, h, w, di, de, seed=h + w + n)
    exact(fused(native, x, illu, e, ac, u8, tiles), stock(native, x, illu, e, ac, u8, tiles))


@gpu
@pytest.mark.parametrize("misalign", ["x", "illu", "e", "illu+e"])
@pytest.mark.parametrize("hw", [(1080, 1920), (400, 600)])
@pytest.mark.parametrize("combo", COMBOS, ids=COMBO_IDS)
def test_misaligned_maps_equal_stock(native, combo, hw, misalign):
    di, de, ac = combo
    x, illu, e = maps(1, *hw, di, de, seed=7, misalign=misalign)
    for u8 in (False, True):
        exact(fused(native, x, illu, e, ac, u8), stock(native, x, illu, e, ac, u8))


@gpu
@pytest.mark.parametrize("combo", COMBOS, ids=COMBO_IDS)
def test_in_place_and_empty_batch(native, combo):
    di, de, ac = combo
    x, illu, e = maps(2, 240, 320, di, de, seed=11)
    want = stock(native, x, illu, e, ac, False)
    got = fused(native, x, illu, e, ac, False, out=x)
    assert got.data_ptr() == x.data_ptr()
    exact(got, want)
    x0, illu0, e0 = maps(0, 64, 64, di, de, seed=1)
    assert fused(native, x0, illu0, e0, ac, False).shape == (0, 3, 64, 64)
    assert fused(native, x0, illu0, e0, ac, True).shape == (0, 64, 64, 3)


@gpu
def test_seeded_sweep_of_shapes_and_grids(native):
    rng = random.Random(2024)
    for case in range(30):
        di, de, ac = COMBOS[rng.randrange(len(COMBOS))]
        n = rng.randint(1, 3)
        h, w = rng.randint(8, 720), rng.randint(8, 720)
        tiles = (rng.randint(1, 16), rng.randint(1, 16))
        if rng.random() < 0.4:     # tile-aligned shapes that may take the vector kernel
            w = max(tiles[0] * 4 * rng.randint(1, 40), 8)
            h = tiles[1] * rng.randint(1, 60)
        misalign = rng.choice(["", "", "illu", "e", "x"])
        u8 = rng.random() < 0.5
        x, illu, e = maps(n, h, w, di, de, seed=case, misalign=misalign)
        got = fused(native, x, illu, e, ac, u8, tiles)
        exact(got, stock(native, x, illu, e, ac, u8, tiles))


def _edge_operands(di, de):
    """A 2 x 3 x 64 x 96 batch with NaN, +-inf, illu = -1e-6 (d = 0) and e large enough that e*e overflows fp16 scattered over it."""
    x, illu, e = maps(2, 64, 96, torch.float32, torch.float32, seed=5)
    g = torch.Generator(device="cpu").manual_seed(6)
    for t, vals in ((x, [float("nan"), float("inf"), -float("inf"), 0.0, 3.0, -2.0]),
                    (illu, [float("nan"), float("inf"), -float("inf"), -1e-6, 0.0, -0.5]),
                    (e, [float("nan"), float("inf"), -float("inf"), 300.0, 260.0, -300.0, 1e4])):
        flat = t.view(-1)
        idx = torch.randint(0, flat.numel(), (flat.numel() // 20,), generator=g)
        pick = torch.randint(0, len(vals), (idx.numel(),), generator=g)
        flat[idx.cuda()] = torch.tensor(vals, device="cuda")[pick.cuda()]
    return x, illu.to(di), e.to(de)


@gpu
@pytest.mark.parametrize("combo", COMBOS, ids=COMBO_IDS)
def test_edge_values_follow_stock(native, combo):
    di, de, ac = combo
    x, illu, e = _edge_operands(di, de)
    big = e.float().abs()
    assert bool(((big >= 256) & torch.isfinite(big)).any())    # finite values whose square overflows fp16 (65504)
    for u8 in (False, True):
        exact(fused(native, x, illu, e, ac, u8), stock(native, x, illu, e, ac, u8))
    r, enh = native.retinex_recombine_typed(x, illu, e, autocast=ac, eps=EPS)
    sr, senh = stock_lines(x, illu, e, ac)
    exact(r, sr)
    exact(enh, senh)


@gpu
@pytest.mark.parametrize("shape,misalign", [((2, 64, 96), ""), ((1, 1080, 1920), ""), ((2, 63, 97), ""), ((2, 64, 96), "e"),
                                            ((2, 64, 96), "illu")], ids=["vec", "vec1080p", "ragged", "e_off", "illu_off"])
@pytest.mark.parametrize("combo", COMBOS, ids=COMBO_IDS)
def test_recombine_typed_equals_eager(native, combo, shape, misalign):
    di, de, ac = combo
    x, illu, e = maps(*shape, di, de, seed=3, misalign=misalign)
    sr, senh = stock_lines(x, illu, e, ac)
    r, enh = native.retinex_recombine_typed(x, illu, e, autocast=ac, eps=EPS)
    exact(r, sr)
    exact(enh, senh)
    r2, enh2 = native.retinex_recombine_typed(x, illu, e, autocast=ac, want_reflectance=False, eps=EPS)
    assert r2 is None
    exact(enh2, senh)
    r3, enh3 = native.retinex_recombine_typed(x, illu, None, eps=EPS)
    assert enh3 is None
    exact(r3, x / (illu + EPS))


@gpu
def test_typed_wrappers_refuse_other_pairs(native):
    x, illu, e = maps(1, 32, 32, torch.float16, torch.bfloat16, seed=1)
    with pytest.raises(TypeError):
        native.retinex_clahe(x, illu, e)
    with pytest.raises(TypeError):
        native.retinex_recombine_typed(x, illu, e)
    with pytest.raises(TypeError):
        native.retinex_clahe(x, illu, e.float())
    with pytest.raises(TypeError):     # x stays f32
        native.retinex_clahe(x.half(), illu.float(), e)


MARGIN = 4096


def _between_nans(t):
    buf = torch.full((t.numel() + 2 * MARGIN,), float("nan"), dtype=t.dtype, device="cuda")
    return buf[MARGIN:MARGIN + t.numel()].view(t.shape).copy_(t), buf


@gpu
@pytest.mark.parametrize("hw,tiles", [((37, 53), (8, 8)), ((403, 601), (16, 16)), ((136, 240), (8, 8)), ((1, 7), (1, 1))])
@pytest.mark.parametrize("combo", COMBOS, ids=COMBO_IDS)
def test_memory_safety_on_awkward_shapes(native, combo, hw, tiles):
    """Inputs between NaN margins (a read outside them would poison the result), outputs between canaries (a write outside
    them would change one)."""
    di, de, ac = combo
    x, illu, e = maps(2, *hw, di, de, seed=9)
    xs, _ = _between_nans(x)
    ils, _ = _between_nans(illu)
    es, _ = _between_nans(e)
    for u8 in (False, True):
        shape = (2, hw[0], hw[1], 3) if u8 else x.shape
        dt = torch.uint8 if u8 else torch.float32
        numel = int(np.prod(shape))
        slab = torch.full((numel + 2 * MARGIN,), 77, dtype=dt, device="cuda")
        out = slab[MARGIN:MARGIN + numel].view(shape)
        fused(native, xs, ils, es, ac, u8, tiles, out=out)
        torch.cuda.synchronize()
        assert bool((slab[:MARGIN] == 77).all()) and bool((slab[MARGIN + numel:] == 77).all())
        exact(out, stock(native, x, illu, e, ac, u8, tiles))
    refl, enh = native.retinex_recombine_typed(xs, ils, es, autocast=ac, eps=EPS)
    sr, senh = stock_lines(x, illu, e, ac)
    exact(refl, sr)
    exact(enh, senh)


# ---- model level: maps captured from the same call ---------------------------------------------------------------------------
class Capture:
    """Wraps models.model._forward_maps (model(x)) or a model's forward_maps (the drivers) and keeps the last maps it returned."""

    def __init__(self, fn):
        self.fn, self.maps = fn, None

    def __call__(self, *a):
        self.maps = self.fn(*a)
        return self.maps


def _network():
    from retinex_image_enhancement_b200.models.model import UP_Retinex
    torch.manual_seed(1)
    return UP_Retinex(use_preact=False, use_aspp=False).cuda().eval()


@gpu
@pytest.mark.parametrize("dt", HALVES, ids=["fp16", "bf16"])
def test_model_call_under_autocast_equals_stock(native, monkeypatch, dt):
    from retinex_image_enhancement_b200.models import model as M
    net = _network()
    cap = Capture(M._forward_maps)
    monkeypatch.setattr(M, "_forward_maps", cap)
    x = torch.rand((2, 3, 128, 192), device="cuda")
    with torch.no_grad(), torch.autocast("cuda", dtype=dt):
        enhanced, refl, illu = net(x)
    illu_c, e_c = cap.maps
    assert (illu_c.dtype, e_c.dtype) == (torch.float32, dt)
    sr, senh = stock_lines(x, illu_c, e_c, True)
    exact(enhanced, senh)
    exact(refl, sr)
    # the decomposition alone, with an illumination map in the autocast dtype
    exact(net.retinex_decompose(x, illu_c.to(dt)), x / (illu_c.to(dt) + EPS))


@gpu
@pytest.mark.parametrize("dt", HALVES, ids=["fp16", "bf16"])
def test_drivers_under_callers_autocast_equal_stock(native, dt):
    from retinex_image_enhancement_b200.enhancers.adaptive_params import AdaptiveParameterAdjuster
    from retinex_image_enhancement_b200.enhancers.simple_enhance import enhance_frames_u8
    net = _network()
    cap = Capture(net.forward_maps)
    net.forward_maps = cap
    x = torch.rand((2, 3, 240, 320), device="cuda")
    with torch.autocast("cuda", dtype=dt):
        out, illu = AdaptiveParameterAdjuster().apply_adaptive_enhancement(net, x, "cuda")
    illu_c, e_c = cap.maps
    assert e_c.dtype == dt and illu is illu_c
    exact(out, stock(native, x, illu_c, e_c, True, False))
    with torch.autocast("cuda", dtype=dt):
        enh8, illu8 = enhance_frames_u8(net, x)
    illu_c, e_c = cap.maps
    exact(enh8, stock(native, x, illu_c, e_c, True, True))
    exact(illu8, native.quantize_u8(illu_c.float().contiguous()))


class AmpStub(torch.nn.Module):
    """Pointwise maps shaped like the real network's under autocast -- illu f32, e in the autocast dtype -- and bit-identical
    whatever the batch composition (cuDNN convolutions are not)."""

    def forward_maps(self, x):
        e = torch.sqrt(x)
        if torch.is_autocast_enabled("cuda"):
            e = e.to(torch.get_autocast_dtype("cuda"))
        return x.mean(dim=1, keepdim=True) * 0.5 + 0.25, e

    def forward(self, x):
        from retinex_image_enhancement_b200.models.model import retinex_recombine
        illu, e = self.forward_maps(x)
        reflectance, enhanced = retinex_recombine(x.contiguous(), illu.contiguous(), e.contiguous())
        return enhanced, reflectance, illu


def _read_png(path):
    from PIL import Image
    return np.asarray(Image.open(path).convert("RGB"))


def _write_pngs(src, count, h, w, seed):
    from PIL import Image
    src.mkdir()
    for i in range(count):
        Image.fromarray(np.random.default_rng(seed + i).integers(0, 90, (h, w, 3), dtype=np.uint8)).save(src / f"f{i}.png")


@gpu
@pytest.mark.parametrize("amp", ["fp16", "bf16"])
def test_batch_and_predict_drivers_with_amp_write_stock_bytes(native, tmp_path, amp):
    from retinex_image_enhancement_b200.enhancers.simple_enhance import (AMP_DTYPES, enhance_batch_images, enhance_single_image,
                                                                         load_image)
    from retinex_image_enhancement_b200.predictors.predict import predict_batch
    src = tmp_path / "in"
    _write_pngs(src, 5, 96, 160, 10)
    stub = AmpStub()
    enhance_batch_images(str(src), str(tmp_path / "batch"), "cuda", model=stub, batch_size=2, amp=amp)
    predict_batch(stub, str(src), str(tmp_path / "pred"), "cuda", batch_size=2, amp=amp)
    for i in range(5):
        low, _ = load_image(str(src / f"f{i}.png"), device="cuda")
        illu, e = stub.forward_maps(low)
        e = e.to(AMP_DTYPES[amp])
        assert np.array_equal(_read_png(tmp_path / "batch" / f"f{i}_enhanced.png"), stock(native, low, illu, e, True, True)[0].cpu().numpy())
        pred = stock_lines(low, illu, e, True)[1]
        assert np.array_equal(_read_png(tmp_path / "pred" / f"f{i}_enhanced.png"), native.quantize_u8(pred)[0].cpu().numpy())
    enhance_single_image(stub, str(src / "f3.png"), str(tmp_path / "single"), "cuda", amp=amp)
    assert np.array_equal(_read_png(tmp_path / "single" / "f3_enhanced.png"), _read_png(tmp_path / "batch" / "f3_enhanced.png"))
    # amp off is today's f32 path: different bytes somewhere in the batch
    enhance_batch_images(str(src), str(tmp_path / "f32"), "cuda", model=stub, batch_size=2)
    assert any(not np.array_equal(_read_png(tmp_path / "f32" / f"f{i}_enhanced.png"), _read_png(tmp_path / "batch" / f"f{i}_enhanced.png"))
               for i in range(5))


@gpu
def test_cli_amp_writes_the_single_image_drivers_bytes(native, tmp_path):
    from PIL import Image

    from retinex_image_enhancement_b200 import cli
    from retinex_image_enhancement_b200.enhancers.simple_enhance import enhance_single_image
    Image.fromarray(np.random.default_rng(4).integers(0, 90, (128, 192, 3), dtype=np.uint8)).save(tmp_path / "p.png")
    torch.manual_seed(21)
    cli.main(["--mode", "enhance", "--input_path", str(tmp_path / "p.png"), "--output_dir", str(tmp_path / "cli"), "--device", "cuda",
              "--amp", "fp16"])
    torch.manual_seed(21)
    net = cli._model("cuda")
    enhance_single_image(net, str(tmp_path / "p.png"), str(tmp_path / "drv"), "cuda", amp="fp16")
    for suffix in ("enhanced", "illumination", "comparison"):
        assert np.array_equal(_read_png(tmp_path / "cli" / f"p_{suffix}.png"), _read_png(tmp_path / "drv" / f"p_{suffix}.png"))
    cli.simple_enhance_main(["--input", str(tmp_path / "p.png"), "--output", str(tmp_path / "cli2"), "--amp", "bf16"])
    assert os.path.exists(tmp_path / "cli2" / "p_enhanced.png")


@gpu
@pytest.mark.parametrize("ac", [False, True], ids=["noac", "ac"])
def test_f32_maps_keep_the_f32_entries(native, ac):
    """f32 / f32 maps are today's call whatever the autocast flag (the kernel is pinned by the profiler test below): the
    result of the stock composition in f32."""
    x, illu, e = maps(2, 240, 320, torch.float32, torch.float32, seed=12)
    for u8 in (False, True):
        exact(fused(native, x, illu, e, ac, u8), stock(native, x, illu, e, False, u8))
    r, enh = native.retinex_recombine_typed(x, illu, e, autocast=ac, eps=EPS)
    sr, senh = stock_lines(x, illu, e, False)
    exact(r, sr)
    exact(enh, senh)


# Run in a child process: a profiler session leaves process-wide tracing state behind, and later sessions of the suite
# (which look for their own kernels in a trace) must not depend on how many ran before them.
PROFILE_CHILD = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
import torch
from torch.profiler import ProfilerActivity, profile
from retinex_image_enhancement_b200 import native
g = torch.Generator(device="cuda").manual_seed(2)
x = torch.rand((2, 3, 1080, 1920), device="cuda", generator=g)
illu = torch.rand((2, 1, 1080, 1920), device="cuda", generator=g) * 0.9 + 0.05
e = torch.rand((2, 3, 1080, 1920), device="cuda", generator=g)
cases = {"f32-f16": (illu, e.half(), True), "f16-f16": (illu.half(), e.half(), True), "f32-f32": (illu, e, True)}
names = {}
for k, (il, ee, ac) in cases.items():
    native.retinex_clahe_u8(x, il, ee, autocast=ac)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        native.retinex_clahe_u8(x, il, ee, autocast=ac)
        torch.cuda.synchronize()
    names[k] = [ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]
print(json.dumps(names))
"""


@gpu
def test_profiler_shows_the_half_map_kernel_and_no_cast(native):
    """The fused autocast call runs the K1 instantiation of its map dtypes and no cast or copy kernel on e; f32 maps keep
    today's kernel."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-s", "-c", PROFILE_CHILD, root], capture_output=True, text=True, cwd=root, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    names = json.loads(r.stdout.strip().splitlines()[-1])
    want = {"f32-f16": "k_hist_lab_vec3<false, true, float, __half, true>",
            "f16-f16": "k_hist_lab_vec3<false, true, __half, __half, true>",
            "f32-f32": "k_hist_lab_vec3<false, true, float, float, false>"}
    for k, kernel in want.items():
        assert any(kernel in n for n in names[k]), (k, names[k])
        assert not any(w in n.lower() for n in names[k] for w in ("copy", "cast", "elementwise")), (k, names[k])
