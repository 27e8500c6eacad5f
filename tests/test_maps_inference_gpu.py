"""Content-aware, multi-scale and predict inference straight from the CNN maps: the Retinex recombination formed inside the last
pass of each mode (upr_retinex_content_aware_typed_*, upr_retinex_multiscale_typed_*, upr_retinex_quantize_typed_u8).

Every result is compared bit for bit with the composition the drivers ran before: the two Retinex lines of models/model.py in
torch eager under torch.autocast("cuda", dtype=e.dtype, enabled=autocast), then content_aware_apply / multiscale_enhance / nothing,
then quantize_u8 for the stored frames and quantize_u8(illu.float()) for the illumination frame."""
import os
import random

import numpy as np
import pytest
import torch

EPS = 1e-6
HALVES = (torch.float16, torch.bfloat16)
COMBOS = [(torch.float32, torch.float32, False)] + [(di, de, ac) for de in HALVES for di in (torch.float32, de) for ac in (False, True)]
COMBO_IDS = [f"{str(di)[6:]}-{str(de)[6:]}-{'ac' if ac else 'noac'}" for di, de, ac in COMBOS]
MODES = ["ca", "ca8", "ms", "ms8", "pred8"]
gpu = pytest.mark.gpu


def _lib():
    import __graft_entry__ as g
    g.ensure_built()
    from retinex_image_enhancement_b200 import native
    return native.lib()


# ---- CPU: status codes (every pointer NULL, so no order of the checks can reach a launch) ------------------------------------
F32, F16, BF16, AC = 0, 1, 2, 1
ENTRIES = {
    "upr_retinex_content_aware_typed_f32": lambda f, di, de, fl, n, h, w: f(None, None, di, None, de, fl, None, n, h, w, EPS, None, 0, None),
    "upr_retinex_content_aware_typed_u8": lambda f, di, de, fl, n, h, w: f(None, None, di, None, de, fl, None, None, n, h, w, EPS, None, 0,
                                                                           None),
    "upr_retinex_multiscale_typed_f32": lambda f, di, de, fl, n, h, w: f(None, None, di, None, de, fl, None, None, None, n, h, w, EPS, None,
                                                                         0, None),
    "upr_retinex_multiscale_typed_u8": lambda f, di, de, fl, n, h, w: f(None, None, di, None, de, fl, None, None, None, None, n, h, w, EPS,
                                                                        None, 0, None),
    "upr_retinex_quantize_typed_u8": lambda f, di, de, fl, n, h, w: f(None, None, di, None, de, fl, None, None, n, h, w, EPS, None),
}


@pytest.mark.parametrize("name", sorted(ENTRIES))
def test_maps_entries_check_their_arguments(name):
    entry, call0 = getattr(_lib(), name), ENTRIES[name]

    def call(di, de, fl, n=1, h=8, w=8):
        return call0(entry, di, de, fl, n, h, w)

    for di, de in ((F32, F16), (F32, BF16), (F16, F16), (BF16, BF16), (F32, F32)):
        for fl in (0, AC):
            assert call(di, de, fl) == -1                     # NULL
            assert call(di, de, fl, n=0) == 0                 # empty batch
    assert call(F32, 3, 0) == -4                              # unknown e dtype
    assert call(5, F16, 0) == -4                              # unknown illu dtype
    assert call(F32, -1, 0) == -4
    assert call(F16, BF16, 0) == -4                           # illu neither f32 nor e's dtype
    assert call(BF16, F16, AC) == -4
    assert call(F16, F32, 0) == -4
    assert call(F32, F16, 2) == -4                            # unknown flag
    assert call(F32, F16, AC | 4) == -4
    assert call(F32, F16, 0, h=0) == -2                       # bad shape, checked first
    assert call(F32, F16, 0, n=-1) == -2
    assert call(F16, BF16, 2, w=0) == -2
    assert call(F16, BF16, 0, n=0) == -4                      # dtypes before the empty-batch rule
    if "multiscale" in name:
        assert call(F32, F16, 0, h=3) == -2                   # no 1/4 scale
        assert call(F16, BF16, 0, w=2, n=0) == -2
    if "quantize" not in name:
        assert call(F32, F16, 0, n=65536) == -2


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
    with torch.autocast("cuda", dtype=e.dtype if e.dtype != torch.float32 else torch.float16, enabled=autocast):
        r = x / (illu + EPS)
        return r, r * e + (1 - r) * (e ** 2)


def stock(native, mode, x, illu, e, ac):
    """The composition the drivers ran before, as a tuple of the entry's results."""
    enh = stock_lines(x, illu, e, ac)[1]
    assert enh.dtype == torch.float32
    illu8 = native.quantize_u8(illu.float().contiguous())
    if mode.startswith("ca"):
        out = native.content_aware_apply(x, enh)
        return (out,) if mode == "ca" else (native.quantize_u8(out), illu8)
    if mode.startswith("ms"):
        out, means, gain = native.multiscale_enhance(x, enh)
        return (out, means, gain) if mode == "ms" else (native.quantize_u8(out), illu8)
    return native.quantize_u8(enh), illu8


def fused(native, mode, x, illu, e, ac, **kw):
    fn = {"ca": native.retinex_content_aware, "ca8": native.retinex_content_aware_u8, "ms": native.retinex_multiscale,
          "ms8": native.retinex_multiscale_u8, "pred8": native.retinex_quantize_u8}[mode]
    r = fn(x, illu, e, autocast=ac, eps=EPS, **kw)
    return r if isinstance(r, tuple) else (r,)


def check(native, mode, x, illu, e, ac, **kw):
    got = fused(native, mode, x, illu, e, ac, **kw)
    want = stock(native, mode, x, illu, e, ac)
    assert len(got) == len(want)
    for g, w in zip(got, want):
        exact(g, w)
    return got


def maps(n, h, w, di, de, seed, misalign=""):
    """x [n,3,h,w] f32 in [0,1), illu in [0.05, 0.95) and e in [0, 1.2) on the GPU; `misalign` names the tensors that start one
    element past an aligned address."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.rand((n, 3, h, w), generator=g)
    illu = (torch.rand((n, 1, h, w), generator=g) * 0.9 + 0.05).to(di)
    e = (torch.rand((n, 3, h, w), generator=g) * 1.2).to(de)
    return [_place(t.cuda(), name in misalign) for name, t in (("x", x), ("illu", illu), ("e", e))]


def _place(t, off):
    if not off:
        return t
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    return buf[1:].view(t.shape).copy_(t)


def _outs(mode, shape, off):
    """out= / out_illu= for the mode, one element off alignment when `off`."""
    n, _, h, w = shape
    if mode in ("ca", "ms"):
        return {"out": _place(torch.empty(shape, device="cuda"), off)}
    return {"out": _place(torch.empty((n, h, w, 3), dtype=torch.uint8, device="cuda"), off),
            "out_illu": _place(torch.empty((n, h, w, 1), dtype=torch.uint8, device="cuda"), off)}


SHAPES = [(2, 1080, 1920), (1, 2160, 3840), (3, 64, 96), (2, 37, 53)]


@gpu
@pytest.mark.parametrize("shape", SHAPES, ids=["2x1080p", "4k", "3x64x96", "ragged"])
@pytest.mark.parametrize("combo", COMBOS, ids=COMBO_IDS)
@pytest.mark.parametrize("mode", MODES)
def test_entry_equals_composition(native, mode, combo, shape):
    di, de, ac = combo
    x, illu, e = maps(*shape, di, de, seed=1)
    check(native, mode, x, illu, e, ac)


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_seeded_sweep_of_shapes_and_batches(native, mode):
    rng = random.Random(7)
    for case in range(30):
        n, h, w = rng.randint(1, 4), rng.randint(4, 300), rng.randint(4, 300)
        if case % 3 == 0:
            h, w = h // 4 * 4 + 4, w // 8 * 8 + 16      # the vector and streaming paths
        di, de, ac = COMBOS[case % len(COMBOS)]
        x, illu, e = maps(n, h, w, di, de, seed=100 + case, misalign=rng.choice(["", "", "x", "e"]))
        check(native, mode, x, illu, e, ac)


@gpu
@pytest.mark.parametrize("hw", [(1080, 1920), (400, 600)], ids=["1080p", "400x600"])
@pytest.mark.parametrize("off", ["x", "illu", "e", "out", "x,illu,e,out"])
@pytest.mark.parametrize("mode", MODES)
def test_misaligned_operands(native, mode, hw, off):
    for di, de, ac in (COMBOS[0], COMBOS[2], COMBOS[7]):
        x, illu, e = maps(2, *hw, di, de, seed=3, misalign=off)
        check(native, mode, x, illu, e, ac, **_outs(mode, x.shape, "out" in off))


@gpu
@pytest.mark.parametrize("combo", COMBOS, ids=COMBO_IDS)
@pytest.mark.parametrize("mode", ["ca", "ms"])
def test_in_place_and_empty_batch(native, mode, combo):
    """out = x at 1080p, where the content-aware chain would otherwise keep luma in `out` between its passes."""
    di, de, ac = combo
    x, illu, e = maps(2, 1080, 1920, di, de, seed=4)
    want = stock(native, mode, x, illu, e, ac)
    got = fused(native, mode, x, illu, e, ac, out=x)
    assert got[0].data_ptr() == x.data_ptr()
    for g, w in zip(got, want):
        exact(g, w)
    for m in (mode, mode + "8"):
        x0, il0, e0 = maps(0, 64, 96, di, de, seed=4)
        for t in fused(native, m, x0, il0, e0, ac):
            assert t.shape[0] == 0
    x0, il0, e0 = maps(0, 64, 96, di, de, seed=4)
    assert fused(native, "pred8", x0, il0, e0, ac)[0].shape == (0, 64, 96, 3)


def _edge_operands(di, de):
    """A 2 x 3 x 64 x 96 batch with NaN, +-inf, illu = -eps (d = 0) and e large enough that e*e overflows fp16."""
    x, illu, e = maps(2, 64, 96, torch.float32, torch.float32, seed=5)
    g = torch.Generator(device="cpu").manual_seed(6)
    for t, vals in ((x, [float("nan"), float("inf"), -float("inf"), 0.0, 3.0, -2.0]),
                    (illu, [float("nan"), float("inf"), -float("inf"), -EPS, 0.0, -0.5]),
                    (e, [float("nan"), float("inf"), -float("inf"), 300.0, 260.0, -300.0, 1e4])):
        flat = t.view(-1)
        idx = torch.randint(0, flat.numel(), (flat.numel() // 20,), generator=g)
        pick = torch.randint(0, len(vals), (idx.numel(),), generator=g)
        flat[idx.cuda()] = torch.tensor(vals, device="cuda")[pick.cuda()]
    return x, illu.to(di), e.to(de)


@gpu
@pytest.mark.parametrize("combo", COMBOS, ids=COMBO_IDS)
@pytest.mark.parametrize("mode", MODES)
def test_edge_values_follow_composition(native, mode, combo):
    di, de, ac = combo
    x, illu, e = _edge_operands(di, de)
    big = e.float().abs()
    assert bool(((big >= 256) & torch.isfinite(big)).any())
    check(native, mode, x, illu, e, ac)
    check(native, mode, x[:, :, :, 1:], illu[:, :, :, 1:], e[:, :, :, 1:], ac)     # the scalar path


MARGIN = 4096


def _between(t, fill):
    buf = torch.full((t.numel() + 2 * MARGIN,), fill, dtype=t.dtype, device="cuda")
    return buf[MARGIN:MARGIN + t.numel()].view(t.shape).copy_(t), buf


@gpu
@pytest.mark.parametrize("hw", [(37, 53), (403, 601), (136, 240), (4, 7)])
@pytest.mark.parametrize("combo", COMBOS, ids=COMBO_IDS)
@pytest.mark.parametrize("mode", MODES)
def test_memory_safety_on_awkward_shapes(native, mode, combo, hw):
    """Inputs between NaN margins (a read outside them would poison the result), outputs and workspace between canaries (a
    write outside them would change one)."""
    di, de, ac = combo
    x, illu, e = maps(2, *hw, di, de, seed=9)
    xs, _ = _between(x, float("nan"))
    ils, _ = _between(illu, float("nan"))
    es, _ = _between(e, float("nan"))
    slabs, kw = [], {}
    for k, t in _outs(mode, x.shape, False).items():
        canary = 77 if t.dtype == torch.uint8 else 7.0
        v, slab = _between(torch.zeros_like(t), canary)
        slabs.append((slab, canary, t.numel()))
        kw[k] = v
    got = fused(native, mode, xs, ils, es, ac, **kw)
    torch.cuda.synchronize()
    for slab, canary, numel in slabs:
        assert bool((slab[:MARGIN] == canary).all()) and bool((slab[MARGIN + numel:] == canary).all())
    for g, w in zip(got, stock(native, mode, x, illu, e, ac)):
        exact(g, w)
    # the workspace: the library's workspace between canaries, as large as the size function asks
    if mode != "pred8":
        size_fn = "upr_saliency_workspace_bytes" if mode.startswith("ca") else "upr_multiscale_workspace_bytes"
        nbytes = getattr(native.lib(), size_fn)(2, *hw)
        slab = torch.full((nbytes + 2 * MARGIN,), 0x5A, dtype=torch.uint8, device="cuda")
        slab[MARGIN:MARGIN + nbytes].zero_()
        ws = slab[MARGIN:MARGIN + nbytes]
        out = torch.empty_like(x)
        if mode.startswith("ca"):
            args = (out.data_ptr(), 2, *hw, EPS, ws.data_ptr(), nbytes)
            entry = "upr_retinex_content_aware_typed_f32"
        else:
            means, gain = torch.empty((2, 3), device="cuda"), torch.empty((2,), device="cuda")
            args = (out.data_ptr(), means.data_ptr(), gain.data_ptr(), 2, *hw, EPS, ws.data_ptr(), nbytes)
            entry = "upr_retinex_multiscale_typed_f32"
        rc = getattr(native.lib(), entry)(xs.data_ptr(), ils.data_ptr(), native.MAP_DTYPES[di], es.data_ptr(), native.MAP_DTYPES[de],
                                          int(ac), *args, torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        torch.cuda.synchronize()
        assert bool((slab[:MARGIN] == 0x5A).all()) and bool((slab[MARGIN + nbytes:] == 0x5A).all())
        exact(out, stock(native, mode.rstrip("8"), x, illu, e, ac)[0])
        assert getattr(native.lib(), entry)(xs.data_ptr(), ils.data_ptr(), native.MAP_DTYPES[di], es.data_ptr(),
                                            native.MAP_DTYPES[de], int(ac), *args[:-1], 8, 0) == -3     # workspace too small


@gpu
@pytest.mark.parametrize("mode", MODES)
def test_repeatable_under_a_busy_second_stream(native, mode):
    """26 x 1080p runs as three chunks on the two side streams: 20 calls give the same bytes while another stream keeps the
    GPU busy."""
    di, de, ac = torch.float32, torch.float16, True
    x, illu, e = maps(26, 1080, 1920, di, de, seed=11)
    first = check(native, mode, x, illu, e, ac)
    side = torch.cuda.Stream()
    a = torch.rand((4096, 4096), device="cuda")
    for _ in range(20):
        with torch.cuda.stream(side):
            for _ in range(4):
                a = a @ a / 4096.0
        for g, w in zip(fused(native, mode, x, illu, e, ac), first):
            exact(g, w)
    torch.cuda.synchronize()


@gpu
def test_wrappers_refuse_other_pairs(native):
    x, illu, e = maps(1, 32, 32, torch.float16, torch.bfloat16, seed=1)
    for mode in MODES:
        with pytest.raises(TypeError):
            fused(native, mode, x, illu, e, False)
    assert not native.maps_supported(x, illu, e)
    assert native.maps_supported(x, illu.float(), e)
    assert not native.maps_supported(x.cpu(), illu.float().cpu(), e.cpu())


# ---- drivers: a stub with forward_maps against the same model with forward_maps hidden ----------------------------------------
class MapsStub(torch.nn.Module):
    """Pointwise maps shaped like the real network's -- illu f32, e in the autocast dtype under autocast -- and bit-identical
    whatever the batch composition."""

    def forward_maps(self, x):
        e = torch.sqrt(x) * 1.1
        if torch.is_autocast_enabled("cuda"):
            e = e.to(torch.get_autocast_dtype("cuda"))
        return x.mean(dim=1, keepdim=True) * 0.5 + 0.2, e

    def forward(self, x):
        from retinex_image_enhancement_b200.models.model import retinex_recombine
        illu, e = self.forward_maps(x)
        reflectance, enhanced = retinex_recombine(x.contiguous(), illu.contiguous(), e.contiguous())
        return enhanced, reflectance, illu


class Hidden(torch.nn.Module):
    """The same model without forward_maps: the drivers take the model(x) path."""

    def __init__(self, inner):
        super().__init__()
        self.inner = inner

    def forward(self, x):
        return self.inner(x)


AMPS = [None, "fp16", "bf16"]


@gpu
@pytest.mark.parametrize("amp", AMPS, ids=["f32", "fp16", "bf16"])
def test_drivers_equal_the_model_call_path(native, amp):
    from retinex_image_enhancement_b200.enhancers.content_aware import ContentAwareEnhancer
    from retinex_image_enhancement_b200.enhancers.multi_scale import MultiScaleEnhancer
    from retinex_image_enhancement_b200.enhancers.simple_enhance import amp_context, enhance_frames_u8
    stub = MapsStub().eval()
    x = torch.rand((3, 3, 240, 320), device="cuda")
    for ms, ca in ((True, False), (False, True), (True, True)):
        with amp_context(amp):
            got = enhance_frames_u8(stub, x, enable_multi_scale=ms, enable_content_aware=ca)
            want = enhance_frames_u8(Hidden(stub), x, enable_multi_scale=ms, enable_content_aware=ca)
        for g, w in zip(got, want):
            exact(g, w)
    for enh in (ContentAwareEnhancer().apply_content_aware_enhancement, MultiScaleEnhancer().apply_multi_scale_enhancement):
        with amp_context(amp):
            got = enh(stub, x, "cuda")
            want = enh(Hidden(stub), x, "cuda")
        exact(got[0], want[0])
        exact(got[1], want[1])
    # CPU operands keep the model(x) path (which then fails on the device-only kernels exactly as before)
    from retinex_image_enhancement_b200.enhancers.adaptive_params import cnn_maps
    assert cnn_maps(stub, x.cpu()) is None
    stub.train()
    assert cnn_maps(stub, x) is None


def _read_png(path):
    from PIL import Image
    return np.asarray(Image.open(path).convert("RGB"))


def _write_pngs(src, count, h, w, seed):
    from PIL import Image
    src.mkdir()
    for i in range(count):
        Image.fromarray(np.random.default_rng(seed + i).integers(0, 90, (h, w, 3), dtype=np.uint8)).save(src / f"f{i}.png")


@gpu
@pytest.mark.parametrize("amp", AMPS, ids=["f32", "fp16", "bf16"])
def test_batch_and_predict_drivers_write_the_model_call_bytes(native, tmp_path, amp):
    from retinex_image_enhancement_b200.enhancers.simple_enhance import enhance_batch_images
    from retinex_image_enhancement_b200.predictors.predict import predict_batch
    src = tmp_path / "in"
    _write_pngs(src, 5, 96, 160, 20)
    stub = MapsStub().eval()
    for tag, model in (("maps", stub), ("call", Hidden(stub))):
        predict_batch(model, str(src), str(tmp_path / f"pred_{tag}"), "cuda", batch_size=2, amp=amp)
        for ms, ca in ((True, False), (False, True)):
            enhance_batch_images(str(src), str(tmp_path / f"b{int(ms)}{int(ca)}_{tag}"), "cuda", model=model, batch_size=2,
                                 enable_multi_scale=ms, enable_content_aware=ca, amp=amp)
    for d in ("pred", "b10", "b01"):
        for i in range(5):
            for suffix in ("enhanced", "illumination", "comparison"):
                assert np.array_equal(_read_png(tmp_path / f"{d}_maps" / f"f{i}_{suffix}.png"),
                                      _read_png(tmp_path / f"{d}_call" / f"f{i}_{suffix}.png")), (d, i, suffix)


# Run in a child process: a profiler session leaves process-wide tracing state behind.
PROFILE_CHILD = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
import torch
from torch.profiler import ProfilerActivity, profile
from retinex_image_enhancement_b200.enhancers.simple_enhance import enhance_frames_u8
from retinex_image_enhancement_b200.predictors.predict import predict_batch
sys.path.insert(0, sys.argv[1] + "/tests")
from test_maps_inference_gpu import MapsStub
from retinex_image_enhancement_b200 import native
stub = MapsStub().eval()
x = torch.rand((2, 3, 1080, 1920), device="cuda")
runs = {"ca": lambda: enhance_frames_u8(stub, x, enable_content_aware=True),
        "ms": lambda: enhance_frames_u8(stub, x, enable_multi_scale=True)}
def pred():
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        il, e = stub.forward_maps(x)
        native.retinex_quantize_u8(x, il, e, autocast=True)
runs["pred"] = pred
names = {}
for k, fn in runs.items():
    fn(); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn(); torch.cuda.synchronize()
    names[k] = [ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]
print(json.dumps(names))
"""


@gpu
def test_profiler_shows_the_map_epilogues_and_no_recombine_or_quantize(native):
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-s", "-c", PROFILE_CHILD, root], capture_output=True, text=True, cwd=root, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    names = json.loads(r.stdout.strip().splitlines()[-1])
    want = {"ca": "k_maps_epilogue_vec<float, float, false, true, upr::AttGain>",
            "ms": "k_maps_epilogue_vec<float, float, false, true, upr::FrameGain>",
            "pred": "k_maps_epilogue_vec<float, __half, true, true, upr::NoGain>"}
    for k, kernel in want.items():
        assert any(kernel in n for n in names[k]), (k, names[k])
        assert not any(w in n for n in names[k] for w in ("k_recombine", "k_quantize_u8", "k_att_gain", "k_gain_clamp")), (k, names[k])
