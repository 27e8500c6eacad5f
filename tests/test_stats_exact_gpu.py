"""Pixel-level checks of the statistics kernels against the CPU oracle.

The statistics kernels reduce a frame to a few numbers, and a loose tolerance on those numbers hides errors confined to a few
pixels.  These tests compare exactly wherever the kernel performs the oracle's operations in the oracle's order, and make the
one kernel that cannot be exact sensitive to single pixels:

  (a) the multi-scale feature maps of the generic path (k_ms_downsample + k_ms_features), all 21 channels, bit for bit, and its
      means within one fp32 ulp of the oracle's fp64 means;
  (b) probe frames through the streaming multi-scale kernel (k_ms_stream): zero frames with a few asymmetric patches whose
      offsets sweep every lane, pixel, row and walking direction of its band / segment grid -- with a CPU proof that one wrong
      pixel moves a mean by at least ten times the tolerance;
  (c) texture TV on dyadic inputs, where every partial sum is exact: per image, batch pair and dynamic weight, exactly;
  (d) texture edge density, exactly, including a frame whose Sobel magnitudes tie with the threshold;
  (e) the brightness histogram over all 2^24 colours.
"""
import numpy as np
import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu

f32 = np.float32


@pytest.fixture(scope="module")
def native():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from retinex_image_enhancement_b200 import native as nat
    assert nat.lib().upr_device_check() == 0
    return nat


def expect_equal(got, want, what):
    """Exact equality (NaN equals NaN), reporting the first differing positions."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    bad = got != want
    if got.dtype.kind == "f":
        bad &= ~(np.isnan(got) & np.isnan(want))
    if bad.any():
        idx = np.argwhere(bad)[:6]
        sel = tuple(idx.T)
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} values differ; first at {idx.tolist()}: "
                             f"got {got[sel].tolist()}, want {want[sel].tolist()}")


def dev(a, offset=0):
    """`a` on the device; offset > 0 places it `offset` floats into a fresh buffer: a contiguous view whose address is not
    16-byte aligned, which sends the kernels down their scalar paths."""
    a = np.ascontiguousarray(a)
    if offset == 0:
        return torch.from_numpy(a).cuda()
    buf = torch.empty(a.size + offset, dtype=torch.float32, device="cuda")
    v = buf[offset:].view(a.shape)
    v.copy_(torch.from_numpy(a))
    assert v.is_contiguous() and v.data_ptr() % 16 != 0
    return v


def fp32_weight(s, cnt, w0=1.0):
    """dyn_weight of upr_stats.cu restated in fp32: clamp(w0 * (1 - 0.8 * s / cnt), 0.1, 5.0), NaN passing through."""
    avg = f32(s) / f32(cnt)
    wv = f32(w0) * (f32(1) - avg * f32(0.8))
    return f32(0.1) if wv < f32(0.1) else (f32(5.0) if wv > f32(5.0) else wv)


def fp32_index_sum(v):
    s = f32(0)
    for t in np.asarray(v, np.float32):
        s = f32(s + t)
    return s


def check_batch_stats(native, x, method, per_image):
    """stats2 = [fp32 sum of the per-image values in index order, float(n)], and the dynamic weight from both the separate
    kernel and the fused one, all exactly."""
    got, stats = native.texture_complexity(x, method, want_batch_stats=True)
    expect_equal(got.cpu().numpy(), per_image, f"{method}: per image (batch-stats call)")
    s, n = fp32_index_sum(per_image), f32(len(per_image))
    expect_equal(stats.cpu().numpy(), np.array([s, n], np.float32), f"{method}: batch stats")
    for w0 in (1.0, 0.7):
        want = np.array(fp32_weight(s, n, w0), np.float32)
        expect_equal(native.dynamic_smooth_weight(stats, w0).cpu().numpy(), want, f"{method}: dynamic weight, w0={w0}")
        _, stats_p, weight = native.texture_weight_peer(x, method, w0, None, 0, 1, 1)
        expect_equal(stats_p.cpu().numpy(), stats.cpu().numpy(), f"{method}: batch stats (fused weight kernel)")
        expect_equal(weight.cpu().numpy(), want, f"{method}: dynamic weight (fused weight kernel), w0={w0}")


# ---- (a) feature maps of the generic path, bit for bit ------------------------------------------------------------------
FEATURE_CASES = [
    (1, 72, 104, 0), (1, 1080, 1920, 0), (1, 101, 67, 0),
    (1, 40, 45, 0), (1, 41, 46, 0), (1, 42, 47, 0), (1, 43, 44, 0),     # every residue of h mod 4 and of w mod 4
    (1, 4, 37, 0), (1, 7, 30, 0), (1, 33, 5, 0), (1, 6, 6, 0),         # quarter image one pixel tall / wide: grad1's len == 1
    (3, 50, 70, 0),                                                     # a batch
    (2, 64, 96, 1), (1, 101, 67, 3),                                    # frames at non-16-byte-aligned addresses
]


@pytest.mark.parametrize("n,h,w,offset", FEATURE_CASES)
def test_feature_maps_bit_exact(native, n, h, w, offset):
    """upr_multiscale_features_f32 (the generic path: bilinear down-sample, then one feature kernel per scale) performs the
    oracle's fp32 operations in the oracle's order (the oracle is built with -ffp-contract=off), so all 21 channels at the three
    scales equal O.multiscale_features bit for bit, at exact and inexact scales (int(101 * 0.25) = 25).  The means of the
    generic path are fp64 sums in another order: within one fp32 ulp of the oracle's fp64 means (the earlier bound, 2e-6
    relative, is about 17 ulp), and the gain equals float32 of the oracle's factor whenever the three means are bit-equal."""
    rng = np.random.default_rng(n * 10007 + h * 101 + w)
    x = rng.random((n, 3, h, w), dtype=np.float32)
    xd = dev(x, offset)
    f1, f2, f3, means, gain = native.multiscale_features(xd)
    got = [f.cpu().numpy() for f in (f1, f2, f3)]
    m_g, g_g = native.multiscale_stats(xd, force_generic=True)
    m_g, g_g = m_g.cpu().numpy(), g_g.cpu().numpy()
    expect_equal(means.cpu().numpy(), m_g, "means of the features entry == force_generic means")
    expect_equal(gain.cpu().numpy(), g_g, "gain of the features entry == force_generic gain")
    for i in range(n):
        want = O.multiscale_features(x[i])
        for s, (g, wnt) in enumerate(zip(got, want)):
            expect_equal(g[i], wnt, f"frame {i}, scale {s}: feature maps")
        m_ref, f_ref = O.multiscale_means(x[i])
        ulp = np.spacing(m_ref.astype(np.float32))
        assert (np.abs(m_g[i].astype(np.float64) - m_ref) <= ulp).all(), (i, m_g[i].tolist(), m_ref.tolist())
        if np.array_equal(m_g[i], m_ref.astype(np.float32)):
            assert g_g[i] == f32(f_ref), (i, float(g_g[i]), f_ref)
    if n == 3:      # the public drop-in returns the same maps
        from retinex_image_enhancement_b200.enhancers.multi_scale import MultiScaleEnhancer
        feats = MultiScaleEnhancer().extract_multi_scale_features(xd)
        for s in range(3):
            expect_equal(feats[s].cpu().numpy(), got[s], f"extract_multi_scale_features, scale {s}")


# ---- (b) probe frames through the streaming kernel -----------------------------------------------------------------------
BAND = 120          # k_ms_stream: 120 counted columns per warp (lanes 1..30, 4 columns each; lanes 0 and 31 are halo)
PATCH = 3
# Largest relative error of a streaming mean on these probe batches, measured on a B200 (1000 W limit): 6.3e-8, about one fp32
# ulp (the rounding of the mean itself; the approximate square roots add far less).  The tolerance keeps a margin of ~5x, and
# the sensitivity proof below holds against the tolerance, not against the smaller error seen.
MS_RTOL = 3e-7


def seg_rows_of(h, w):
    """Row-segment height of k_ms_stream's launch: 64 rows, doubled while the frame has more than 4096 (band, segment) cells."""
    bands, seg = -(-w // BAND), 64
    while bands * -(-h // seg) > 4096 and seg < h:
        seg *= 2
    return seg


def probe_batch(h, w, frames, k, seed):
    """[frames,3,h,w] zero frames with asymmetric 3x3 patches (random values in [0.25, 1), different in every channel):
      * up to k in full (band, segment) cells, at most one per cell.  Patch j of the batch sits at column offset j % 120 and
        row offset j % seg inside its cell, in a segment whose parity alternates every L = max(120, seg) patches: 2L patches put
        every column residue (every lane, every pixel of a lane, the pixels next to both halo lanes) and every row residue into
        even (downward) and odd (upward) segments.  Offsets 118-119 and seg-2, seg-1 straddle the band / segment boundary;
      * up to 4 in partial cells (the last band, the last segment), clipped into the frame;
      * on the four corners and, in frames of at least 64 x 64, at four points of the borders.
    -> (x, patches [(frame, y0, x0, full cell, column offset, row offset, segment parity)])"""
    rng = np.random.default_rng(seed)
    seg = seg_rows_of(h, w)
    bands, segs = -(-w // BAND), -(-h // seg)
    full = {p: [(b, s) for s in range(segs) if s % 2 == p and (s + 1) * seg <= h for b in range(w // BAND)] for p in (0, 1)}
    partial = [(b, s) for s in range(segs) for b in range(bands) if (b + 1) * BAND > w or (s + 1) * seg > h]
    period = max(BAND, seg)
    borders = [(0, 0), (0, w - PATCH), (h - PATCH, 0), (h - PATCH, w - PATCH)]
    if h >= 64 and w >= 64:
        borders += [(0, w // 2), (h - PATCH, w // 3), (h // 2, 0), (h // 3, w - PATCH)]
    x = np.zeros((frames, 3, h, w), np.float32)
    patches = []

    def put(f, y0, x0, *info):
        x[f, :, y0:y0 + PATCH, x0:x0 + PATCH] = rng.uniform(0.25, 1.0, (3, PATCH, PATCH)).astype(np.float32)
        patches.append((f, y0, x0) + info)

    j = 0
    for f in range(frames):
        pools = {p: [full[p][i] for i in rng.permutation(len(full[p]))] for p in (0, 1)}
        for _ in range(k):
            par = (j // period) % 2
            if not pools[par]:
                par = 1 - par
            if not pools[par]:
                break
            b, s = pools[par].pop()
            put(f, s * seg + j % seg, b * BAND + j % BAND, True, j % BAND, j % seg, s % 2)
            j += 1
        for i in rng.permutation(len(partial))[:4]:
            b, s = partial[i]
            oy, ox = int(rng.integers(seg)), int(rng.integers(BAND))
            put(f, min(s * seg + oy, h - PATCH), min(b * BAND + ox, w - PATCH), False, ox, oy, s % 2)
        for y0, x0 in borders:
            put(f, y0, x0, False, None, None, None)
    return x, patches


def scales_reached(y, xx):
    """Scales a pixel feeds at exact 1/2 and 1/4 scales: every pixel is in a 2x2 block of the half image, only the centre 2x2
    of each 4x4 block is sampled by the quarter image."""
    return (0, 1, 2) if (y % 4 in (1, 2) and xx % 4 in (1, 2)) else (0, 1)


PROBE_CASES = [
    # (h, w, frames, k): every case takes the streaming path (h, w multiples of 4, aligned, at most 4096 cells)
    (1080, 1924, 4, 64),      # 17 bands, the last one holding a single counted lane (w = 120 * 16 + 4); last segment even
    (200, 484, 2, 64),        # last segment (rows 192-199) odd-indexed, walking upwards; single-lane last band again
    (8, 244, 2, 64),          # h / 4 == 2
    (196, 8, 2, 64),          # w / 4 == 2
    (4320, 7680, 4, 64),      # 8K: 128-row segments; 64 of the 2176 cells per frame
]


@pytest.mark.parametrize("h,w,frames,k", PROBE_CASES)
def test_stream_probe_frames(native, h, w, frames, k):
    """k_ms_stream (sqrt.approx and FMA: not exact) on probe frames, the whole batch in one call so that the frame index
    (blockIdx.y) varies too: each mean within MS_RTOL of O.multiscale_means.  The test proves its own sensitivity: for a
    sample of patches, one pixel raised by 1/64 in its three channels in the oracle's input moves the oracle's mean by at
    least 10x the tolerance at every scale that pixel feeds -- so a kernel that gets a single pixel of a patch wrong (a
    swapped neighbour, a luma weight on the wrong channel, a missing border doubling) fails.  (All three channels: raising
    one channel of a pixel lowers the gradients of brighter neighbours, and on a few pixels the two nearly cancel.)  The
    patches are asymmetric and differ per channel, because |grad| is even and equal channels would hide a weight on the
    wrong channel."""
    seg = seg_rows_of(h, w)
    x, patches = probe_batch(h, w, frames, k, seed=h * 7 + w)
    if (h, w) in ((1080, 1924), (4320, 7680)):
        assert seg == (128 if h == 4320 else 64)
        full = [p for p in patches if p[3]]
        for what, idx, mod in (("column", 4, BAND), ("row", 5, seg)):
            for par in (0, 1):
                seen = {p[idx] for p in full if p[6] == par}
                assert seen == set(range(mod)), f"{what} residues missing from {('even', 'odd')[par]} segments"
    xd = dev(x)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        m, g = native.multiscale_stats(xd)
        torch.cuda.synchronize()
    assert any("k_ms_stream" in e.name for e in prof.events()), "the streaming kernel was not launched"
    m_gen, _ = native.multiscale_stats(xd, force_generic=True)
    m, g, m_gen = m.cpu().numpy(), g.cpu().numpy(), m_gen.cpu().numpy()
    if h * w < 4e6:
        # the approximate square roots show in the last bits; at 8K the means are so small and the patches so few that both
        # paths round to the same fp32 values, and the kernel's launch (above) is the evidence
        assert not np.array_equal(m.view(np.uint32), m_gen.view(np.uint32)), "streaming and generic means are bit-equal"
    worst = 0.0
    refs = []
    for i in range(frames):
        m_ref, f_ref = O.multiscale_means(x[i])
        refs.append(m_ref)
        rel = np.abs(m[i].astype(np.float64) - m_ref) / m_ref
        worst = max(worst, float(rel.max()))
        assert (rel <= MS_RTOL).all(), (i, rel.tolist())
        assert abs(float(g[i]) - f_ref) <= 2e-7 * f_ref
    print(f"probe {h}x{w}: worst relative error of a mean {worst:.3g}")
    # sensitivity: one pixel of a sampled patch, +1/64 in its three channels
    rng = np.random.default_rng(h + w)
    sample = [patches[i] for i in rng.choice(len(patches), 3 if h * w > 4e6 else 6, replace=False)]
    for f, y0, x0, *_ in sample:
        ys, xs = np.meshgrid(np.arange(y0, y0 + PATCH), np.arange(x0, x0 + PATCH), indexing="ij")
        quarter = [(int(a), int(b)) for a, b in zip(ys.ravel(), xs.ravel()) if len(scales_reached(a, b)) == 3]
        other = [(int(a), int(b)) for a, b in zip(ys.ravel(), xs.ravel()) if len(scales_reached(a, b)) == 2]
        picks = [quarter[rng.integers(len(quarter))]] + ([other[rng.integers(len(other))]] if other else [])
        for y, xx in picks:
            xp = x[f].copy()
            xp[:, y, xx] += f32(1 / 64)
            moved = np.abs(O.multiscale_means(xp)[0] - refs[f])
            for s in scales_reached(y, xx):
                assert moved[s] >= 10 * MS_RTOL * refs[f][s], (f, y, xx, s, moved[s] / (MS_RTOL * refs[f][s]))


# ---- (c) TV, exact on dyadic inputs ----------------------------------------------------------------------------------------
def tv_expected(k, c, h, w):
    """The kernel's TV of the frames k / 4096 (k integer): every |a - b| is a multiple of 2^-12, so the kernel's fp32 partial
    sums of up to 4 terms and its fp64 totals are exact; it rounds each mean once to fp32 and adds the two in fp32."""
    out = []
    for kk in k:
        sh = int(np.abs(np.diff(kk, axis=2)).sum(dtype=np.int64))
        sv = int(np.abs(np.diff(kk, axis=1)).sum(dtype=np.int64))
        with np.errstate(invalid="ignore", divide="ignore"):
            mh = f32(np.float64(sh / 4096.0) / np.float64(c * h * (w - 1)))
            mv = f32(np.float64(sv / 4096.0) / np.float64(c * (h - 1) * w))
        out.append(f32(mh + mv))
    return np.array(out, np.float32)


TV_CASES = [
    # (n, c, h, w, offset)
    (2, 3, 64, 96, 0), (3, 1, 40, 64, 0), (2, 4, 36, 52, 0),        # vector path: w % 4 == 0, aligned
    (2, 3, 33, 31, 0), (1, 1, 7, 9, 0), (2, 4, 5, 3, 0),            # scalar path: w % 4 != 0
    (2, 3, 64, 96, 1), (1, 1, 40, 64, 2),                           # scalar path: w % 4 == 0 at an unaligned address
    (1, 3, 2160, 3840, 0), (1, 3, 4320, 7680, 0), (4, 3, 540, 960, 0),
    (2, 3, 1, 40, 0), (2, 1, 40, 1, 0), (1, 3, 1, 1, 0),            # h == 1 / w == 1: NaN, like torch's mean of an empty slice
    (3, 4, 1, 64, 0),
]


@pytest.mark.parametrize("n,c,h,w,offset", TV_CASES)
def test_tv_exact(native, n, c, h, w, offset):
    """texture_complexity(.., "tv") on dyadic frames equals the int64 restatement exactly: per image, the batch pair and the
    dynamic weight.  (The oracle's texture_tv rounds its double sum once, so it is not the expectation here.)"""
    rng = np.random.default_rng(n * 31 + c * 7 + h + w)
    k = rng.integers(0, 4097, (n, c, h, w), dtype=np.int32)
    x = k.astype(np.float32) / f32(4096)
    assert np.array_equal((x * f32(4096)).astype(np.int32), k)
    want = tv_expected(k, c, h, w)
    if h == 1 or w == 1:
        assert np.isnan(want).all()
    xd = dev(x, offset)
    expect_equal(native.texture_complexity(xd, "tv").cpu().numpy(), want, "tv per image")
    check_batch_stats(native, xd, "tv", want)


# ---- (d) edge density, exact -----------------------------------------------------------------------------------------------
def sobel_np(g):
    """|Sobel| of one gray plane in fp32, reflect-101 borders: upr_stats.cu's sobel_mag in NumPy (same operation order)."""
    p = g
    for ax in (0, 1):     # reflect-101; a length-1 axis reflects onto itself
        pad = [(0, 0), (0, 0)]
        pad[ax] = (1, 1)
        p = np.pad(p, pad, mode="reflect" if g.shape[ax] > 1 else "edge")
    a, b, cc = p[:-2, :-2], p[:-2, 1:-1], p[:-2, 2:]
    d, f = p[1:-1, :-2], p[1:-1, 2:]
    gg, hh, k = p[2:, :-2], p[2:, 1:-1], p[2:, 2:]
    gx = ((cc - a) + f32(2) * (f - d)) + (k - gg)
    gy = ((gg - a) + f32(2) * (hh - b)) + (k - cc)
    return np.sqrt(gx * gx + gy * gy)


def assert_mean_clear_of_fp32_ties(x):
    """Precondition of exactness: the threshold is float32(mean magnitude) * 1.5, and the kernel and the oracle sum the n
    magnitudes in different orders.  Both fp64 sums of n non-negative terms, and the division by n, are within
    (n + 1) * 2^-53 relative of the exact mean, so if the oracle's mean is farther than twice that from every fp32 rounding
    boundary, both round to the same fp32 threshold."""
    _, means = O.texture_edge_density(x, want_mean=True)
    n = x.shape[2] * x.shape[3]
    for m in means:
        if m == 0.0:
            continue
        f = np.float32(m)
        lo, hi = np.nextafter(f, f32(-np.inf)), np.nextafter(f, f32(np.inf))
        bounds = ((np.float64(f) + np.float64(lo)) / 2, (np.float64(f) + np.float64(hi)) / 2)
        margin = max(1e-15, 2 * (n + 1) * 2.0 ** -53) * m
        assert min(abs(m - b) for b in bounds) > margin, (m, bounds)


EDGE_CASES = [
    # (n, c, h, w): the shapes of test_ops_gpu.test_texture_vs_oracle, then single rows / columns, 2 x 2, c in {1, 3, 4}, 4K
    (2, 3, 64, 96), (3, 1, 33, 31), (1, 3, 640, 640), (5, 3, 7, 9), (2, 4, 2, 2),
    (2, 3, 1, 50), (2, 1, 50, 1), (1, 4, 1, 7), (3, 1, 2, 2), (2, 3, 2, 2), (1, 1, 1, 1),
    (3, 4, 96, 128), (1, 3, 2160, 3840),
]


@pytest.mark.parametrize("n,c,h,w", EDGE_CASES)
def test_edge_density_exact(native, n, c, h, w):
    """Per pixel, sobel_mag performs the oracle's separately rounded fp32 operations, and the threshold is the same
    float(mean) * 1.5f, so the count -- and the per-image density, batch pair and weight -- equal the oracle's bit for bit."""
    x = np.random.default_rng(n * 1009 + c * 101 + h * 7 + w).random((n, c, h, w), dtype=np.float32)
    assert_mean_clear_of_fp32_ties(x)
    want = O.texture_edge_density(x)
    xd = dev(x)
    expect_equal(native.texture_complexity(xd, "edge_density").cpu().numpy(), want, "edge density per image")
    check_batch_stats(native, xd, "edge_density", want)


def tie_frame():
    """64 x 64, one channel, vertical stripes of period 8 (values k / 4): gy = 0 and |gx| = 4 |v[x+1] - v[x-1]| in {0..4}, the
    mean magnitude is exactly 2, the threshold exactly 3, and 512 pixels sit exactly on it (found by a CPU search over
    periodic dyadic patterns)."""
    prof = np.array([1.0, 1.0, 0.5, 0.75, 0.0, 0.0, 1.0, 1.0], np.float32)
    return np.ascontiguousarray(np.broadcast_to(np.tile(prof, 8), (1, 1, 64, 64))).astype(np.float32)


def test_edge_density_threshold_tie(native):
    """A frame where some magnitudes equal the threshold: counting with >= would give another result, so this checks the
    strict > of the reference (loss.py: edges > threshold)."""
    x = tie_frame()
    m = sobel_np(x[0, 0])
    thr = f32(m.astype(np.float64).mean()) * f32(1.5)
    n_gt, n_ge = int((m > thr).sum()), int((m >= thr).sum())
    assert n_ge != n_gt and (n_gt, n_ge) == (1024, 1536)
    want = np.array([n_gt / m.size], np.float32)
    expect_equal(O.texture_edge_density(x), want, "oracle, tie frame")
    for offset in (0, 1):
        xd = dev(x, offset)
        expect_equal(native.texture_complexity(xd, "edge_density").cpu().numpy(), want, "edge density, tie frame")


def test_sobel_restatement_matches_oracle():
    """The NumPy Sobel used for the tie frame counts like the oracle on random frames (so its >= count is meaningful)."""
    for h, w in ((33, 31), (2, 2), (64, 96)):
        x = np.random.default_rng(h + w).random((1, 1, h, w), dtype=np.float32)
        m = sobel_np(x[0, 0])
        thr = f32(m.astype(np.float64).mean()) * f32(1.5)
        assert O.texture_edge_density(x)[0] == f32((m > thr).sum() / m.size)


# ---- (e) brightness histogram over every colour ----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cube_f32():
    """Every sRGB colour once as a [1,3,4096,4096] f32 frame of k / 255 (r slowest), and its u8 planes."""
    i = np.arange(1 << 24, dtype=np.uint32)
    rgb = np.stack([i >> 16, (i >> 8) & 255, i & 255]).astype(np.uint8)
    k255 = np.arange(256, dtype=np.float32) / f32(255)
    return k255[rgb].reshape(1, 3, 4096, 4096), rgb


@pytest.mark.parametrize("layout", ["vector", "offset", "ragged"])
def test_brightness_hist_every_colour(native, cube_f32, layout):
    """All 2^24 colours through upr_brightness_hist_f32: the float4 path ("vector"), the scalar path at an unaligned address
    ("offset") and on a 4095 x 4097 frame holding 2^24 - 1 of them ("ragged").  Expectation: np.bincount of O.gray_u8, which
    test_gray_exhaustive_vs_cv2 pins to cv2 over the same cube."""
    x, rgb = cube_f32
    if layout == "ragged":
        x = np.ascontiguousarray(x.reshape(3, -1)[:, :4095 * 4097].reshape(1, 3, 4095, 4097))
        rgb = rgb[:, :4095 * 4097]
    want = np.bincount(O.gray_u8(rgb), minlength=256)
    got = native.brightness_hist(dev(x, 1 if layout == "offset" else 0)).cpu().numpy()[0]
    expect_equal(got.astype(np.int64), want.astype(np.int64), "histogram")
