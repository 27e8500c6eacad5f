"""Seeded random-shape sweeps of the hot-path ops against the oracle (GPU).  The parametrised tests pin the named shapes and the
edges that were thought of; these sweep (shape, batch, tile grid, clip limit, content kind) combinations nobody picked by hand --
ragged widths, frames smaller than a tile grid, single rows / columns where the reference allows them."""
import numpy as np
import pytest
import torch

from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def native():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from retinex_image_enhancement_b200 import native as nat
    assert nat.lib().upr_device_check() == 0
    return nat


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


KINDS = ("uniform", "dark", "ramp", "const")


def _frames(rng, n, h, w):
    return np.concatenate([O.kat_input(int(rng.integers(1 << 30)), h, w, KINDS[int(rng.integers(len(KINDS)))]) for _ in range(n)])


def test_clahe_random_shapes_grids_and_clips(native):
    """CLAHE-in-Lab bit-exact against the oracle on 40 random (n, h, w, tiles, clip) combinations: the vector kernels (tile width a
    multiple of 4, no padding) and the generic ones (OpenCV's reflect-101 padding when the grid does not divide the frame)."""
    rng = np.random.default_rng(20260)
    for case in range(40):
        tx, ty = int(rng.integers(1, 13)), int(rng.integers(1, 13))
        if case % 2 == 0:      # divisible, 4-px aligned tiles: the fast path
            h, w = ty * int(rng.integers(2, 40)), tx * 4 * int(rng.integers(1, 30))
        else:
            h, w = int(rng.integers(max(2, ty), 300)), int(rng.integers(max(2, tx), 400))
        n = int(rng.integers(1, 4))
        clip = float(rng.choice([0.0, 0.5, 1.0, 2.0, 3.7, 40.0]))
        x = _frames(rng, n, h, w)
        got = native.clahe_lab(dev(x), clip_limit=clip, tiles=(tx, ty)).cpu().numpy()
        for i in range(n):
            ref = O.clahe_lab(x[i], clip, (tx, ty))
            assert np.array_equal(got[i], ref[0]), (case, n, h, w, tx, ty, clip, float(np.abs(got[i] - ref[0]).max()))


def test_multiscale_and_texture_random_shapes(native):
    """Multi-scale means / gain and both texture statistics on 40 random shapes (streaming kernel when h, w are multiples of 4,
    generic kernels otherwise), 2e-6 relative against the oracle; edge density exactly."""
    rng = np.random.default_rng(20261)
    for case in range(40):
        if case % 2 == 0:
            h, w = 4 * int(rng.integers(2, 120)), 4 * int(rng.integers(2, 160))
        else:
            h, w = int(rng.integers(4, 300)), int(rng.integers(4, 500))
        n = int(rng.integers(1, 4))
        x = _frames(rng, n, h, w)
        xd = dev(x)
        m, g = native.multiscale_stats(xd)
        tv = native.texture_complexity(xd, "tv").cpu().numpy()
        ed = native.texture_complexity(xd, "edge_density").cpu().numpy()
        m, g = m.cpu().numpy(), g.cpu().numpy()
        for i in range(n):
            m_ref, f_ref = O.multiscale_means(x[i:i + 1])
            np.testing.assert_allclose(m[i], m_ref, rtol=2e-6, atol=1e-7, err_msg=str((case, n, h, w)))
            assert abs(float(g[i]) - f_ref) <= 2e-7 * f_ref + 6e-8, (case, n, h, w)
            np.testing.assert_allclose(tv[i:i + 1], O.texture_tv(x[i:i + 1]), rtol=2e-6, atol=1e-7, err_msg=str((case, n, h, w)))
            assert ed[i] == O.texture_edge_density(x[i:i + 1])[0], (case, n, h, w)


def test_content_aware_random_shapes(native):
    """Saliency / attention maps and the fused apply on 30 random shapes (packed kernel for w % 8 == 0, h, w >= 16; the general
    kernel otherwise), full maps against the oracle."""
    rng = np.random.default_rng(20262)
    for case in range(30):
        if case % 2 == 0:
            h, w = int(rng.integers(16, 260)), 8 * int(rng.integers(2, 70))
        else:
            h, w = int(rng.integers(3, 200)), int(rng.integers(3, 300))
        n = int(rng.integers(1, 4))
        x = _frames(rng, n, h, w)
        enh = rng.random((n, 3, h, w), dtype=np.float32) * np.float32(1.2)
        xd = dev(x)
        sal, att = native.saliency(xd).cpu().numpy(), native.attention(xd).cpu().numpy()
        out = native.content_aware_apply(xd, dev(enh)).cpu().numpy()
        for i in range(n):
            s_ref, a_ref = O.saliency(x[i:i + 1]), O.attention(x[i:i + 1])
            np.testing.assert_allclose(sal[i:i + 1], s_ref, rtol=0, atol=1e-6, err_msg=str((case, n, h, w)))
            np.testing.assert_allclose(att[i:i + 1], a_ref, rtol=0, atol=2e-6, err_msg=str((case, n, h, w)))
            np.testing.assert_allclose(out[i:i + 1], O.attention_apply(enh[i], a_ref), rtol=0, atol=2e-6, err_msg=str((case, n, h, w)))


def test_fused_retinex_clahe_and_u8_boundaries_random_shapes(native):
    """upr_retinex_clahe_f32 (+ its u8-output form) and the packed u8 CLAHE entry on 30 random shapes / grids: bit-exact against the
    oracle's recombination followed by its CLAHE-in-Lab, resp. against the oracle on the same bytes."""
    rng = np.random.default_rng(20263)
    for case in range(30):
        tx, ty = int(rng.integers(1, 9)), int(rng.integers(1, 9))
        if case % 3 != 2:
            h, w = ty * int(rng.integers(2, 40)), tx * 4 * int(rng.integers(1, 30))
        else:
            h, w = int(rng.integers(max(2, ty), 200)), int(rng.integers(max(2, tx), 300))
        n = int(rng.integers(1, 3))
        clip = float(rng.choice([0.0, 1.0, 2.0, 5.0]))
        x = _frames(rng, n, h, w)
        illu = (rng.random((n, 1, h, w), dtype=np.float32) * np.float32(0.9) + np.float32(0.05)).astype(np.float32)
        e = rng.random((n, 3, h, w), dtype=np.float32)
        got = native.retinex_clahe(dev(x), dev(illu), dev(e), clip_limit=clip, tiles=(tx, ty)).cpu().numpy()
        got8 = native.retinex_clahe_u8(dev(x), dev(illu), dev(e), clip_limit=clip, tiles=(tx, ty)).cpu().numpy()
        x8 = (rng.integers(0, 256, (n, h, w, 3))).astype(np.uint8)
        out8 = native.clahe_lab_u8(dev(x8), clip_limit=clip, tiles=(tx, ty)).cpu().numpy()
        for i in range(n):
            _refl, enh = O.retinex_recombine(x[i:i + 1], illu[i:i + 1], e[i:i + 1])
            ref = O.clahe_lab(enh[0], clip, (tx, ty))[0]
            assert np.array_equal(got[i], ref), (case, n, h, w, tx, ty, clip)
            ref8 = np.rint(ref * 255.0).astype(np.uint8).transpose(1, 2, 0)      # ref is k / 255 exactly: the stored byte is k
            assert np.array_equal(got8[i], ref8), (case, n, h, w, tx, ty, clip)
            want8 = O.clahe_lab((x8[i].astype(np.float32) / np.float32(255.0)).transpose(2, 0, 1), clip, (tx, ty))[0]
            assert np.array_equal(out8[i], np.rint(want8 * 255.0).astype(np.uint8).transpose(1, 2, 0)), (case, n, h, w, tx, ty, clip)


def test_letterbox_random_geometry(native):
    """The --max_size letterbox (down-scaling) on 30 random (frame, target) pairs: bit-exact against the reference recipe run by
    OpenCV on the host (oracle/cv2_chain.letterbox_ref)."""
    pytest.importorskip("cv2")
    from oracle import cv2_chain
    from retinex_image_enhancement_b200.utils.letterbox import letterbox_tensor
    rng = np.random.default_rng(20264)
    for case in range(30):
        h, w = int(rng.integers(40, 900)), int(rng.integers(40, 1200))
        new_shape = int(rng.integers(32, max(33, min(h, w))))
        x = rng.random((3, h, w), dtype=np.float32)
        ref, ratio, pad = cv2_chain.letterbox_ref(x, new_shape, auto=True, scaleup=False)
        got, ratio2, pad2 = letterbox_tensor(torch.from_numpy(x).cuda(), new_shape=new_shape, auto=True, scaleup=False)
        assert tuple(got.shape) == ref.shape and np.array_equal(got.cpu().numpy(), ref), (case, h, w, new_shape)
        assert ratio == ratio2 and tuple(pad) == tuple(pad2)


def test_loss_kernels_random_shapes(native):
    """SURVEY 8f N3: the smoothness loss + gradient and the three enhanced-image losses + gradients on 24 random shapes against
    the NumPy restatements of the reference's loss modules (themselves pinned to the reference's autograd, tests/test_oracle_pin)."""
    rng = np.random.default_rng(20265)
    for case in range(24):
        b = int(rng.integers(1, 5))
        h, w = int(rng.integers(16, 200)), int(rng.integers(16, 260))
        ci = int(rng.choice([1, 3]))
        illu = rng.random((b, ci, h, w), dtype=np.float32)
        low = rng.random((b, 3, h, w), dtype=np.float32) * np.float32(0.5)
        enh = rng.random((b, 3, h, w), dtype=np.float32)
        lam, alpha = float(rng.choice([1.0, 10.0])), float(rng.choice([0.5, 1.0]))
        loss, _lh, _lv, grad = O.edge_smooth_loss(illu, low, lam, alpha)
        loss3, g = native.edge_smooth_loss(dev(illu), dev(low), lam, alpha)
        assert abs(float(loss3[0]) - float(loss)) <= 2e-6 * abs(float(loss)) + 1e-12, (case, b, ci, h, w)
        assert np.abs(g.cpu().numpy() - grad).max() <= 2e-6 * np.abs(grad).max() + 1e-12, (case, b, ci, h, w)
        (l_exp, l_col, l_spa), grads = O.enhanced_image_losses(enh, low)
        losses, saved = native.enhanced_image_losses(dev(enh), dev(low))
        for k, want in enumerate((l_exp, l_col, l_spa)):
            assert abs(float(losses[k]) - float(want)) <= 3e-6 * abs(float(want)) + 1e-12, (case, k, b, h, w)
            up = torch.zeros(3, device="cuda"); up[k] = 1.0
            got = native.enhanced_image_losses_grad(dev(enh), dev(low), saved, up).cpu().numpy()
            assert np.abs(got - grads[k]).max() <= 3e-6 * np.abs(grads[k]).max() + 1e-12, (case, k, b, h, w)
