"""GPU parity of upr_clahe_lab_f32 (through the C ABI) against the CPU oracle and the golden vectors."""
import hashlib

import numpy as np
import pytest
import torch

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


def run_clahe(native, x_np, clip=2.0, tiles=(8, 8)):
    x = torch.from_numpy(np.ascontiguousarray(x_np)).cuda()
    out = native.clahe_lab(x, clip, tiles)
    hist, lut, lab = native.clahe_debug(x.shape, tiles)
    torch.cuda.synchronize()
    return out.cpu().numpy(), hist.cpu().numpy(), lut.cpu().numpy(), lab.cpu().numpy()


def compare(native, x_np, clip=2.0, tiles=(8, 8)):
    out, hist, lut, lab = run_clahe(native, x_np, clip, tiles)
    for i in range(x_np.shape[0]):
        ref, taps = O.clahe_lab(x_np[i], clip, tiles, taps=True)
        assert np.array_equal(lab[i], taps["lab"]), f"Lab intermediate differs (frame {i})"
        assert np.array_equal(hist[i], taps["hist"]), f"histograms differ (frame {i})"
        assert np.array_equal(lut[i], taps["lut"]), f"LUTs differ (frame {i})"
        assert np.array_equal(out[i], ref[0]), f"output differs (frame {i}): {np.abs(out[i]-ref[0]).max()}"
    return out


def test_tables_match_oracle(native):
    t, o = native.tables(), O.tables()
    assert np.array_equal(t["gamma"], o["gamma"])
    assert np.array_equal(t["cbrt"], o["cbrt"][:2048])
    assert np.array_equal(t["ify"], o["ify"]) and np.array_equal(t["y"], o["y"])
    assert np.array_equal(t["invgamma"], o["invgamma"])


def test_golden_kats(native, golden):
    for rec in golden["clahe"]:
        x = O.kat_input(rec["seed"], rec["h"], rec["w"], rec["kind"])
        out = torch.from_numpy(x).cuda()
        out = native.clahe_lab(out).cpu().numpy()
        assert sha(out) == rec["sha_out"], rec


@pytest.mark.parametrize("shape,kind", [
    ((400, 600), "uniform"), ((400, 600), "dark"), ((1080, 1920), "uniform"), ((1080, 1920), "dark"),
    ((1080, 1920), "ramp"), ((1080, 1920), "const"), ((2160, 3840), "dark"), ((403, 601), "uniform"),
    ((400, 601), "dark"), ((401, 600), "uniform"), ((256, 256), "uniform"), ((640, 640), "dark"),
    ((64, 128), "uniform"), ((17, 23), "uniform"), ((9, 9), "dark"), ((8, 8), "uniform"), ((1024, 1000), "uniform"),
    ((1024, 1024), "ramp"), ((64, 4096), "uniform"), ((4320, 7680), "dark"), ((4320, 7680), "uniform"),
])
def test_against_oracle(native, shape, kind):
    compare(native, O.kat_input(shape[0] * 7 + shape[1] + len(kind), shape[0], shape[1], kind))


def test_batch_frames_are_independent(native):
    xs = np.concatenate([O.kat_input(40 + i, 360, 640, k) for i, k in enumerate(["uniform", "dark", "ramp", "const", "dark"])])
    compare(native, xs)


def test_other_clip_and_grids(native):
    x = O.kat_input(50, 320, 512, "uniform")
    for clip, tiles in [(4.0, (4, 4)), (1.0, (16, 8)), (40.0, (8, 8)), (0.0, (8, 8)), (2.0, (2, 2)), (3.0, (32, 32))]:
        compare(native, x, clip, tiles)


def test_out_of_range_and_special_values(native):
    rng = np.random.default_rng(60)
    x = (rng.random((1, 3, 128, 256), dtype=np.float32) * 3 - 1).astype(np.float32)  # negatives and > 1 wrap mod 256
    x[0, 0, 0, :8] = [np.nan, np.inf, -np.inf, 1e10, -1e10, 8421504.5, 1.0, 0.0]
    x[0, 1, 1, :4] = [1.5, -0.5, 254.9999 / 255, 1e-45]
    compare(native, x)


def test_in_place_and_empty(native):
    x = torch.from_numpy(O.kat_input(61, 256, 512, "dark")).cuda()
    ref = native.clahe_lab(x).clone()
    native.clahe_lab(x, out=x)
    assert torch.equal(x, ref)
    empty = torch.empty((0, 3, 64, 64), device="cuda")
    assert native.clahe_lab(empty).shape == (0, 3, 64, 64)


def test_argument_errors(native):
    with pytest.raises(RuntimeError):
        native.clahe_lab(torch.zeros(1, 3, 8, 8))           # CPU tensor: no CPU path
    with pytest.raises(ValueError):
        native.clahe_lab(torch.zeros(1, 4, 8, 8, device="cuda"))
    with pytest.raises(TypeError):
        native.clahe_lab(torch.zeros(1, 3, 8, 8, device="cuda", dtype=torch.float16))
    with pytest.raises(native.UprError):
        native.clahe_lab(torch.zeros(1, 3, 8, 8, device="cuda"), tiles=(0, 8))


def test_adjuster_drop_in(native):
    from retinex_image_enhancement_b200.enhancers.adaptive_params import AdaptiveParameterAdjuster
    adj = AdaptiveParameterAdjuster()
    x = O.kat_input(2, 400, 600, "dark")
    out = adj.apply_clahe_enhancement(torch.from_numpy(x))
    assert not out.is_cuda and out.shape == (1, 3, 400, 600)
    assert np.array_equal(out.numpy(), O.clahe_lab(x))
    out3 = adj.apply_clahe_enhancement(torch.from_numpy(x[0]))   # [3,H,W] accepted like the reference
    assert torch.equal(out3, out)


def test_full_size_properties(native):
    """64 x 1080p (the bench workload): per-frame results equal the single-frame call, constant frames stay
    constant, histogram mass equals the pixel count."""
    g = torch.Generator(device="cuda").manual_seed(1000)
    x = torch.rand((16, 3, 1080, 1920), device="cuda", generator=g)
    x[1::2] *= 0.3
    x[3] = 0.3
    out = native.clahe_lab(x)
    hist, lut, _ = native.clahe_debug(x.shape, want_lab=False)
    assert int(hist.sum()) == 16 * 1080 * 1920 and bool((hist.sum(-1) == 240 * 135).all())
    for i in (0, 3, 7, 15):
        assert torch.equal(native.clahe_lab(x[i:i + 1].clone()), out[i:i + 1])
    assert float(out[3].std()) == 0.0
    assert float(out.min()) >= 0.0 and float(out.max()) <= 1.0


# ---- strip / pass geometry of the column-owner histogram kernel --------------------------------------------------
def test_tiles_wider_than_the_byte_counters_allow(native):
    """One row of a 65536-px tile is 64 four-pixel items per thread (> 63 = 252 px, the budget of the private byte counters
    between flushes): such shapes must leave the vector path.  Strip geometry at the budget (tile 64512 px wide: 63 passes of
    256 columns, one-row strips) stays on it."""
    for w in (8 * 65536, 2 * 64512):
        tiles = (8, 1) if w == 8 * 65536 else (2, 1)
        x = O.kat_input(400, 4, w, "const")        # worst case: every pixel of a thread lands in one bin
        x[0, :, 2:, : w // 2] = O.kat_input(401, 2, w // 2, "dark")[0]
        compare(native, x, 2.0, tiles)


@pytest.mark.parametrize("n,h,w,tiles", [(1, 1080, 1920, (8, 8)), (3, 480, 640, (8, 8)), (2, 256, 1024, (4, 2)), (5, 64, 64, (8, 8)),
                                          (1, 2160, 3840, (16, 16)), (2, 96, 2048, (1, 3))])
def test_persistent_map_kernel_shapes(native, n, h, w, tiles):
    """Work-queue geometry of the persistent map kernel: cells narrower/wider than the CTA, single-row cells, strips."""
    x = np.concatenate([O.kat_input(300 + i, h, w, ("uniform", "dark", "ramp")[i % 3]) for i in range(n)])
    compare(native, x, 2.0, tiles)


# ---- fused Retinex recombination + CLAHE -----------------------------------------------------------------
@pytest.mark.parametrize("n,h,w,tiles", [(2, 1080, 1920, (8, 8)), (3, 400, 600, (8, 8)), (1, 403, 601, (8, 8)), (2, 64, 96, (4, 2)),
                                          (1, 2160, 3840, (8, 8))])
def test_retinex_clahe_fused_equals_composition(native, n, h, w, tiles):
    """upr_retinex_clahe_f32 == upr_retinex_recombine_f32 -> upr_clahe_lab_f32, bit for bit (vector path; generic path on ragged
    shapes), also in place (out = x), and == the oracle's recombination + CLAHE on a small case."""
    rng = np.random.default_rng(h + w)
    x = np.concatenate([O.kat_input(800 + i, h, w, ("dark", "uniform")[i % 2]) for i in range(n)])
    e = rng.random((n, 3, h, w), dtype=np.float32)
    illu = (rng.random((n, 1, h, w), dtype=np.float32) * 0.9 + 0.05).astype(np.float32)
    xd, ed, id_ = (torch.from_numpy(a).cuda() for a in (x, e, illu))
    _, enh = native.retinex_recombine(xd, id_, ed, want_reflectance=False)
    ref = native.clahe_lab(enh, 2.0, tiles)
    got = native.retinex_clahe(xd, id_, ed, 2.0, tiles)
    assert torch.equal(got, ref)
    inplace = xd.clone()
    native.retinex_clahe(inplace, id_, ed, 2.0, tiles, out=inplace)
    assert torch.equal(inplace, ref)
    if h * w <= 400 * 600:
        _, e_ref = O.retinex_recombine(x[:1], illu[:1], e[:1])
        assert np.array_equal(got[:1].cpu().numpy(), O.clahe_lab(e_ref, 2.0, tiles))


@pytest.mark.parametrize("n,h,w,tiles", [(1, 64, 4096, (2, 2)), (2, 48, 2400, (2, 4)), (1, 32, 1200, (1, 1)), (3, 40, 152, (2, 2)),
                                          (1, 2160, 3840, (2, 2))])
def test_column_passes_and_partial_occupancy(native, n, h, w, tiles):
    """Tiles wider than 1024 px are walked in passes of 256 four-pixel columns (2048-px tiles: 2 passes; 1200: 2, the second
    one partial); narrow tiles leave most threads of the CTA without a column (76-px tiles: 19 columns x 13 rows = 247 owners).
    f32, packed u8 and fused-Retinex instantiations of the same kernel."""
    rng = np.random.default_rng(n * h + w)
    x = np.concatenate([O.kat_input(330 + i, h, w, ("uniform", "dark", "ramp")[i % 3]) for i in range(n)])
    compare(native, x, 2.0, tiles)
    x8 = torch.from_numpy(np.ascontiguousarray((x * 255).astype(np.uint8).transpose(0, 2, 3, 1))).cuda()
    out8 = native.clahe_lab_u8(x8, 2.0, tiles).cpu().numpy()
    for i in range(n):
        ref = O.clahe_lab(x8[i].cpu().numpy().transpose(2, 0, 1)[None].astype(np.float32) / np.float32(255.0), 2.0, tiles)
        assert np.array_equal(out8[i].transpose(2, 0, 1).astype(np.float32) / np.float32(255.0), ref[0])
    e = rng.random((n, 3, h, w), dtype=np.float32)
    illu = (rng.random((n, 1, h, w), dtype=np.float32) * 0.9 + 0.05).astype(np.float32)
    xd, ed, id_ = (torch.from_numpy(a).cuda() for a in (x, e, illu))
    got = native.retinex_clahe(xd, id_, ed, 2.0, tiles).cpu().numpy()
    _, e_ref = O.retinex_recombine(x, illu, e)
    for i in range(n):
        assert np.array_equal(got[i:i + 1], O.clahe_lab(e_ref[i:i + 1], 2.0, tiles))


def test_retinex_clahe_u8_output(native):
    """upr_retinex_clahe_f32_u8 == upr_retinex_clahe_f32 followed by save_image's truncating cast (vector path; generic path on
    ragged shapes)."""
    rng = np.random.default_rng(77)
    for n, h, w in ((2, 1080, 1920), (3, 400, 600), (1, 403, 601)):
        x = np.concatenate([O.kat_input(840 + i, h, w, ("dark", "uniform")[i % 2]) for i in range(n)])
        e = rng.random((n, 3, h, w), dtype=np.float32)
        illu = (rng.random((n, 1, h, w), dtype=np.float32) * 0.9 + 0.05).astype(np.float32)
        xd, ed, id_ = (torch.from_numpy(a).cuda() for a in (x, e, illu))
        ref = native.retinex_clahe(xd, id_, ed)
        want = (ref.clamp(0, 1) * 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()
        assert torch.equal(native.retinex_clahe_u8(xd, id_, ed), want)


def misaligned(t):
    """A contiguous copy of t whose data starts one element past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    view = buf[1:].view(t.shape)
    view.copy_(t)
    return view


@pytest.mark.parametrize("which", ["x", "illu", "e"])
@pytest.mark.parametrize("h,w", [(1080, 1920), (400, 600)])
def test_retinex_clahe_misaligned_operand(native, h, w, which):
    """One operand one float past 16-byte alignment: the fused call runs the generic histogram kernel on a shape of the vector
    path.  f32 and u8 outputs bit-identical to upr_retinex_recombine_f32 -> upr_clahe_lab_f32 / upr_clahe_lab_f32_u8."""
    rng = np.random.default_rng(h * w)
    x = np.concatenate([O.kat_input(860 + i, h, w, ("dark", "uniform")[i % 2]) for i in range(2)])
    ops = {"x": x, "e": rng.random((2, 3, h, w), dtype=np.float32),
           "illu": (rng.random((2, 1, h, w), dtype=np.float32) * 0.9 + 0.05).astype(np.float32)}
    ops = {k: torch.from_numpy(a).cuda() for k, a in ops.items()}
    ops[which] = misaligned(ops[which])
    assert ops[which].data_ptr() % 16 == 4
    _, enh = native.retinex_recombine(ops["x"], ops["illu"], ops["e"], want_reflectance=False)
    assert torch.equal(native.retinex_clahe(ops["x"], ops["illu"], ops["e"]), native.clahe_lab(enh))
    assert torch.equal(native.retinex_clahe_u8(ops["x"], ops["illu"], ops["e"]), native.clahe_lab_f32_u8(enh))


def test_second_device_same_process(native):
    """One process driving two GPUs: per-device kernel attributes (dynamic shared memory) and workspaces."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    x = torch.from_numpy(O.kat_input(2, 400, 600, "dark"))
    a = native.clahe_lab(x.to("cuda:0"))
    with torch.cuda.device(1):
        b = native.clahe_lab(x.to("cuda:1"))
        m1, g1 = native.multiscale_stats(x.to("cuda:1"))
        att1 = native.attention(x.to("cuda:1"))
    assert torch.equal(a.cpu(), b.cpu())
    m0, g0 = native.multiscale_stats(x.to("cuda:0"))
    assert torch.equal(m0.cpu(), m1.cpu()) and torch.equal(native.attention(x.to("cuda:0")).cpu(), att1.cpu())
