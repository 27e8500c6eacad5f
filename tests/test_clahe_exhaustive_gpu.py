"""Exhaustive checks of the CLAHE-in-Lab colour path against the CPU oracle.

The sampled tests of test_clahe_gpu.py reach the colour arithmetic only through whatever random content produces.  These
tests enumerate it instead:

  (a) every sRGB colour through K1 (quantise -> sRGB->Lab -> histograms -> LUTs), on every kernel path and entry point;
  (b) every (L', a, b) triple through K3 (Lab->sRGB of the map kernel), fed to the map kernel alone;
  (c) the bilinear LUT interpolation and its rounding ties, with chosen LUTs, on cell geometries of both map kernels;
  (d) the floats on both sides of every quantisation threshold k/255 and the special values, through every quantising kernel.

Everything is compared exactly, except the saliency / attention maps, which keep the tolerances of test_ops_gpu.py.
"""
import numpy as np
import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu

N24 = 1 << 24
K255 = np.arange(256, dtype=np.float32) / np.float32(255)     # k / 255.f: what the f32 entries return for channel value k


@pytest.fixture(scope="module")
def native():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from retinex_image_enhancement_b200 import native as nat
    assert nat.lib().upr_device_check() == 0
    return nat


def expect_equal(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    bad = got != want
    if bad.any():
        idx = np.argwhere(bad)[:6]
        sel = tuple(idx.T)
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} values differ; first at {idx.tolist()}: "
                             f"got {got[sel].tolist()}, want {want[sel].tolist()}")


@pytest.fixture(scope="module")
def cube():
    """Every sRGB colour once, planar [3, 2^24] u8: in natural order (r slowest, the layout of test_oracle_pin.cube) and in
    one seeded pixel permutation (neighbouring pixels of a 4-pixel group, a tile and a cell then hold unrelated colours)."""
    i = np.arange(N24, dtype=np.uint32)
    natural = np.stack([i >> 16, (i >> 8) & 255, i & 255]).astype(np.uint8)
    perm = np.random.default_rng(2024).permutation(N24)
    return {"natural": natural, "permuted": np.ascontiguousarray(natural[:, perm])}


@pytest.fixture(scope="module")
def cube_lab(cube):
    return {order: O.rgb2lab_u8(rgb) for order, rgb in cube.items()}


# ---- (a) every sRGB colour -> Lab, histograms, LUTs, output (K1) -------------------------------------------------------
_oracle_cache = {}


def oracle_clahe_of_lab(lab, key, tiles):
    """(hist, lut, sRGB u8 planes) of the oracle's CLAHE of the Lab planes `lab` [3,h,w]; the last few results are kept."""
    if key not in _oracle_cache:
        if len(_oracle_cache) >= 2:
            _oracle_cache.pop(next(iter(_oracle_cache)))
        l2, hist, lut = O.clahe_u8(lab[0], 2.0, tiles, taps=True)
        _oracle_cache[key] = (hist, lut, O.lab2rgb_u8(np.stack([l2, lab[1], lab[2]])))
    return _oracle_cache[key]


@pytest.mark.parametrize("entry", ["clahe_lab", "clahe_lab_u8", "clahe_lab_f32_u8"])
@pytest.mark.parametrize("shape,tiles", [
    ((4096, 4096), (8, 8)),      # 512-px tiles: the vector kernels
    ((4096, 4096), (16, 16)),    # the largest grid of the vector kernels
    ((4096, 4096), (2, 2)),      # 2048-px tiles: the histogram kernel walks them in two passes of 256 four-pixel columns
    ((4096, 4096), (1, 1)),      # one 4096-px tile: four passes
    ((4095, 4097), (8, 8)),      # 2^24 - 1 colours on a padded shape: the generic kernels
])
@pytest.mark.parametrize("order", ["natural", "permuted"])
def test_every_srgb_colour_through_k1(native, cube, cube_lab, order, shape, tiles, entry):
    """Each of the 2^24 colours once per frame: the device's Lab planes equal O.rgb2lab_u8 pixel for pixel (the oracle's
    conversion is pinned to cv2 over the same cube in test_oracle_pin.py), and histograms, LUTs and the result equal the
    oracle's.  The f32 entries read k / 255.f, which the quantiser maps back to k."""
    h, w = shape
    rgb = cube[order][:, :h * w].reshape(3, h, w)
    lab_ref = cube_lab[order][:, :h * w].reshape(3, h, w)
    if entry == "clahe_lab_u8":
        x = torch.from_numpy(np.ascontiguousarray(rgb.transpose(1, 2, 0))[None]).cuda()
    else:
        x = torch.from_numpy(K255[rgb][None]).cuda()
    out = getattr(native, entry)(x, 2.0, tiles)
    hist, lut, lab = native.clahe_debug((1, 3, h, w), tiles)
    torch.cuda.synchronize()
    del x
    expect_equal(lab[0].cpu().numpy(), lab_ref, "Lab planes")
    hist_ref, lut_ref, want = oracle_clahe_of_lab(lab_ref, (order, shape, tiles), tiles)
    expect_equal(hist[0].cpu().numpy(), hist_ref, "histograms")
    expect_equal(lut[0].cpu().numpy(), lut_ref, "LUTs")
    out = out[0].cpu().numpy()
    if entry == "clahe_lab":
        expect_equal(out, K255[want], "f32 result")
    else:
        expect_equal(out, want.transpose(1, 2, 0), "u8 result")


# ---- (b) every (L', a, b) triple -> sRGB (K3) ------------------------------------------------------------------------
def identity_luts(n_tiles):
    return np.ascontiguousarray(np.broadcast_to(np.arange(256, dtype=np.uint8), (1, n_tiles, 256)))


@pytest.mark.parametrize("shape", [(4096, 4096), (4097, 4096)])
def test_every_lab_triple_through_k3(native, shape):
    """Lab planes that enumerate all 2^24 (L, a, b) triples, identity LUTs (lut[i] = i: non-decreasing and ending at 255, like
    every LUT CLAHE builds), so that L' = L: the map kernel's table arithmetic equals O.lab2rgb_u8 on every triple, including
    the (a, b) pairs that no sRGB colour produces.  4096 x 4096 takes the persistent vector kernel, 4097 x 4096 (padded: the
    last row repeats the first 4096 triples) the generic one."""
    h, w = shape
    i = np.arange(h * w, dtype=np.uint32) % N24
    lab = np.stack([i >> 16, (i >> 8) & 255, i & 255]).astype(np.uint8).reshape(3, h, w)
    lut = identity_luts(64)
    assert np.array_equal(O.clahe_map_u8(lab[0], lut[0]), lab[0])
    out = native.clahe_map_only(torch.from_numpy(lab[None]).cuda(), torch.from_numpy(lut).cuda(), (8, 8))
    expect_equal(out[0].cpu().numpy(), K255[O.lab2rgb_u8(lab)], "f32 result")


# ---- (c) bilinear interpolation and rounding (K3) ----------------------------------------------------------------------
def make_luts(kind, tiles, seed):
    """[tiles_y * tiles_x, 256] u8 LUTs that CLAHE itself could build (non-decreasing, lut[255] = 255)."""
    tx_n, ty_n = tiles
    nt = tx_n * ty_n
    ty, tx = np.divmod(np.arange(nt), tx_n)
    grey = np.arange(256)[None, :]
    rng = np.random.default_rng(seed)
    if kind == "random":      # sorted random bytes
        lut = np.sort(rng.integers(0, 256, (nt, 256)), axis=1)
        lut[:, -1] = 255
    elif kind == "step":      # 0 below a random grey level, 255 from it on: neighbours average to k + 0.5 in many places
        lut = np.where(grey >= rng.integers(1, 256, nt)[:, None], 255, 0)
    elif kind == "chessboard":
        # identity + 0 / 1 in a chessboard: horizontal and vertical neighbours differ by one, the four LUTs around a tile corner
        # sum to 4 i + 2, so xa = 0.5 (with ya = 0 or 0.5) and ya = 0.5 (with xa = 0) are exact .5 ties
        lut = np.minimum(grey + ((tx + ty) % 2)[:, None], 255)
    else:                     # "odd": neighbours differ by 3 across and 5 down (mod 16): ties on the tile edges, not corners
        lut = np.minimum(grey + ((3 * tx + 5 * ty) % 16)[:, None], 255)
    assert (np.diff(lut, axis=1) >= 0).all() and (lut[:, -1] == 255).all()
    return lut.astype(np.uint8)


_lab_dev = {}


@pytest.mark.parametrize("kind", ["random", "step", "chessboard", "odd"])
@pytest.mark.parametrize("shape,tiles", [
    ((4096, 4096), (8, 8)),      # 512-px tiles: power-of-two weights, exact xa = ya = 0.5 at tile corners
    ((4096, 4096), (16, 16)),
    ((4320, 3840), (8, 8)),      # 480 x 540 tiles: inexact weights, products that round
    ((2048, 8192), (2, 2)),      # 4096-px interior cells: twice the width of the 512-thread CTA
    ((2048, 8192), (1, 1)),      # two 4096-px cells
    ((65536, 256), (16, 16)),    # 16-px tiles: 8-px border cells, 4096-row cells
    ((4095, 4097), (8, 8)),      # padded: generic kernel
    ((4000, 4194), (7, 5)),      # padded, odd grid
    ((4096, 4096), (32, 32)),    # more tiles than the vector kernel holds: generic kernel
])
def test_interpolation_and_rounding(native, cube_lab, shape, tiles, kind):
    """Lab planes of the permuted cube through chosen LUTs: the result is exactly O.lab2rgb_u8(O.clahe_map_u8(L, lut), a, b)."""
    h, w = shape
    lab = cube_lab["permuted"][:, :h * w].reshape(3, h, w)
    if shape not in _lab_dev:
        _lab_dev.clear()
        _lab_dev[shape] = torch.from_numpy(lab[None]).cuda()
    lut = make_luts(kind, tiles, seed=h + w + 31 * tiles[0] + tiles[1])
    out = native.clahe_map_only(_lab_dev[shape], torch.from_numpy(lut[None]).cuda(), tiles)
    l2 = O.clahe_map_u8(lab[0], lut, tiles)
    want = O.lab2rgb_u8(np.stack([l2, lab[1], lab[2]]))
    expect_equal(out[0].cpu().numpy(), K255[want], "f32 result")


# ---- (d) quantiser edges ------------------------------------------------------------------------------------------------
def edge_values():
    """Every k / 255.f with the 64 floats on each side of it, and the special values of the quantiser."""
    k = np.arange(256, dtype=np.float32) / np.float32(255)
    vals, lo, hi = [k], k, k
    for _ in range(64):
        lo, hi = np.nextafter(lo, np.float32(-np.inf)), np.nextafter(hi, np.float32(np.inf))
        vals += [lo, hi]

    def ulps(c, n=4):
        c = np.float32(c)
        out = [c]
        for d in (np.float32(-np.inf), np.float32(np.inf)):
            v = c
            for _ in range(n):
                v = np.nextafter(v, d)
                out.append(v)
        return out

    bits = [0x00000000, 0x80000000,                          # +-0
            0x00000001, 0x80000001, 0x007FFFFF, 0x807FFFFF,  # subnormals
            0x00800000, 0x80800000,                          # smallest normals
            0x7F800000, 0xFF800000,                          # +-inf
            0x7FC00000, 0xFFC00000, 0x7F800001, 0xFF800001,  # NaNs: quiet, negative, signalling, payloads
            0x7FBFFFFF, 0x7FFFFFFF, 0xFFFFFFFF, 0x7FC12345]
    special = [np.array(bits, np.uint32).view(np.float32)]
    special += [np.array(ulps(c), np.float32) for c in (1.0, 2.0 ** 23 / 255, 2.0 ** 24 / 255, 2.0 ** 31 / 255,
                                                         -2.0 ** 31 / 255, 256.0 / 255)]
    special += [np.array([1e10, -1e10, 1.5, -0.5, 2.0, -1.0], np.float32)]
    return np.concatenate(vals + special)


def in_range(v):
    """The vector kernels' test: the bit pattern is at most that of 1.0f, i.e. +0 <= v <= 1 (-0 and NaN excluded)."""
    return v.view(np.uint32) <= np.uint32(0x3F800000)


@pytest.fixture(scope="module")
def edge_frame():
    """[1, 3, 256, 256] f32 of the edge values, laid out in 4-pixel groups (12 values: R0..R3 G0..G3 B0..B3, what the vector
    kernels test at once): every in-range value in each channel inside groups that are entirely in range, and every
    out-of-range value alone at each of the 12 positions of a group whose other 11 values are in range.  Such groups are
    paired with an in-range group, first or second, so that out-of-range values visit all 24 positions of the 8-pixel groups
    of the saliency kernel as well.  Rows hold 64 groups, so groups never straddle a row."""
    v = edge_values()
    inr, outr = v[in_range(v)], v[~in_range(v)]
    rng = np.random.default_rng(77)
    full = [np.roll(inr, r) for r in (0, 4, 8)]             # each in-range value as R, G and B
    full = np.concatenate(full + [rng.choice(inr, (-sum(map(len, full))) % 12)]).reshape(-1, 12)
    if len(full) % 2:
        full = np.concatenate([full, rng.choice(inr, (1, 12))])
    alone = rng.choice(inr, (len(outr) * 12, 12))
    alone[np.arange(len(alone)), np.tile(np.arange(12), len(outr))] = np.repeat(outr, 12)
    partner = rng.choice(inr, alone.shape)
    m = np.arange(len(alone))
    first = ((m // 12 + m) % 2 == 0)[:, None, None]     # value j at position p leads its pair when j + p is even
    pairs = np.where(first, np.stack([alone, partner], 1), np.stack([partner, alone], 1))
    groups = np.concatenate([full, pairs.reshape(-1, 12)])
    h, w = 256, 256
    assert len(groups) <= h * w // 4
    groups = np.concatenate([groups, rng.choice(inr, (h * w // 4 - len(groups), 12))])
    frame = np.stack([groups[:, 0:4].ravel(), groups[:, 4:8].ravel(), groups[:, 8:12].ravel()]).reshape(1, 3, h, w)
    assert np.isin(v.view(np.uint32), frame.view(np.uint32)).all()
    return np.ascontiguousarray(frame)


LAYOUTS = {"vector": (256, 256), "ragged": (255, 253)}


def edge_input(edge_frame, layout):
    h, w = LAYOUTS[layout]
    return np.ascontiguousarray(edge_frame[:, :, :h, :w])


@pytest.mark.parametrize("layout", ["vector", "ragged"])
def test_quantiser_edges_clahe(native, edge_frame, layout):
    """clahe_lab on the edge values: Lab planes equal O.rgb2lab_u8(O.quantize_u8(x)) (numpy's (x*255).astype(uint8)), and
    histograms, LUTs and result equal the oracle's.  "vector": 32-px tiles, the magic-add fast path and its range test on
    each 4-pixel group; "ragged": the generic kernel."""
    x = edge_input(edge_frame, layout)
    out = native.clahe_lab(torch.from_numpy(x).cuda())
    hist, lut, lab = native.clahe_debug(x.shape)
    ref, taps = O.clahe_lab(x, taps=True)
    expect_equal(lab[0].cpu().numpy(), O.rgb2lab_u8(O.quantize_u8(x[0])), "Lab planes")
    expect_equal(lab[0].cpu().numpy(), taps["lab"], "Lab planes (oracle taps)")
    expect_equal(hist[0].cpu().numpy(), taps["hist"], "histograms")
    expect_equal(lut[0].cpu().numpy(), taps["lut"], "LUTs")
    expect_equal(out.cpu().numpy(), ref, "result")


@pytest.mark.parametrize("layout", ["vector", "ragged"])
def test_quantiser_edges_other_kernels(native, edge_frame, layout):
    """The same values through the other quantising kernels, at the tolerances of their own tests: brightness histogram
    (exact), saliency / attention (1e-6 / 2e-6; "vector" is w % 8 == 0, the packed kernel with its 24-value range test),
    letterbox without resize (exactly quantise / 255) and save_image's quantiser (exactly numpy's clip-and-cast)."""
    x = edge_input(edge_frame, layout)
    h, w = LAYOUTS[layout]
    xd = torch.from_numpy(x).cuda()
    expect_equal(native.brightness_hist(xd).cpu().numpy()[0].astype(np.uint32), O.brightness_hist(x), "brightness histogram")
    np.testing.assert_allclose(native.saliency(xd).cpu().numpy(), O.saliency(x), rtol=0, atol=1e-6)
    # attention divides by luma(x) + 0.1: a NaN pixel has a NaN luma, and how NaN enters the min / max normalisation is no
    # question of the quantiser -- those pixels read 0 here, every other edge value stays
    xa = np.where(np.isnan(x), np.float32(0), x)
    np.testing.assert_allclose(native.attention(torch.from_numpy(xa).cuda()).cpu().numpy(), O.attention(xa), rtol=0, atol=2e-6)
    lb = native.letterbox(xd, (h, w), 0, 0, (h, w))
    expect_equal(lb.cpu().numpy(), O.quantize_u8(x).astype(np.float32) / np.float32(255), "letterbox")
    with np.errstate(invalid="ignore"):
        q_ref = (np.clip(x, 0, 1) * np.float32(255)).astype(np.uint8)
    expect_equal(native.quantize_u8(xd).cpu().numpy(), q_ref.transpose(0, 2, 3, 1), "quantize_u8, 3 channels")
    expect_equal(native.quantize_u8(xd[:, 1:2].contiguous()).cpu().numpy(), q_ref[:, 1:2].transpose(0, 2, 3, 1),
                 "quantize_u8, 1 channel")
