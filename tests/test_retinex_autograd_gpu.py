"""The two Retinex lines of models/model.py:405-413 and :442 under autograd: the fused forward and gradient kernels
(upr_retinex_recombine_maps / upr_retinex_recombine_grad behind models.model._RetinexFn) against eager torch autograd through
the stock expressions, bit for bit, with f32, fp16 and bf16 maps, with and without CUDA autocast."""
import copy
import itertools
import re

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from retinex_image_enhancement_b200.models import model as M

EPS = M.EPSILON
MAPS = (torch.float32, torch.float16, torch.bfloat16)
gpu = pytest.mark.gpu


def stock(x, illu, e):
    """The reference's own expressions (models/model.py:412, :442)."""
    r = x / (illu + EPS)
    return r, (None if e is None else r * e + (1 - r) * (e ** 2))


def exact(got, want):
    if want is None:
        assert got is None
        return
    assert got is not None and got.dtype == want.dtype and got.shape == want.shape
    torch.testing.assert_close(got, want, rtol=0, atol=0, equal_nan=True)


def operands(n, h, w, dtype, seed, device, misalign=False):
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.rand((n, 3, h, w), generator=g)
    illu = (torch.rand((n, 1, h, w), generator=g) * 0.9 + 0.05).to(dtype)
    e = torch.rand((n, 3, h, w), generator=g).to(dtype)
    out = []
    for t in (x, illu, e):
        t = t.to(device)
        if misalign:   # contiguous, but one element past an aligned address: the scalar kernels
            buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=device)
            t = buf[1:].view(t.shape).copy_(t)
        out.append(t)
    return out


def upstream(like, seed, scale=1.0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return ((torch.rand(like.shape, generator=g) - 0.5) * scale).to(like.device)


def run(fn, x, illu, e, x_grad, up, autocast, g_enh, g_refl):
    """Forward through fn(x, illu, e) -> (R, enhanced | None), backward from the chosen outputs.
    -> (R, enhanced, x.grad, illu.grad, e.grad, grad_fn of R)."""
    x = x.detach().clone().requires_grad_(x_grad)
    illu = illu.detach().clone().requires_grad_()
    e = None if e is None else e.detach().clone().requires_grad_()
    amp = illu.dtype if illu.dtype != torch.float32 else torch.float16
    with torch.autocast("cuda", dtype=amp, enabled=autocast):
        r, enh = fn(x, illu, e)
    outs, grads = [], []
    if up in ("refl", "both"):
        outs.append(r), grads.append(g_refl)
    if up in ("enh", "both"):
        outs.append(enh), grads.append(g_enh)
    torch.autograd.backward(outs, grads)
    return r, enh, x.grad, illu.grad, (None if e is None else e.grad), r.grad_fn


def fused(x, illu, e):
    if e is None:
        return M.retinex_decompose(x, illu), None
    return M.retinex_recombine(x, illu, e)


def check_case(x, illu, e, x_grad, up, autocast, scale=1.0):
    g_enh, g_refl = upstream(x, 11, scale), upstream(x, 12, scale)
    got = run(fused, x, illu, e, x_grad, up, autocast, g_enh, g_refl)
    want = run(stock, x, illu, e, x_grad, up, autocast, g_enh, g_refl)
    assert type(got[5]).__name__ == "_RetinexFnBackward"
    for g, w in zip(got[:5], want[:5]):
        exact(g, w)
    return got


# ------------------------------------------------------------------------------------------------------------------
# CPU: the pinned formulas (the differentiable torch ops that backward(create_graph=True) evaluates) against autograd
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", MAPS)
@pytest.mark.parametrize("up", ["enh", "refl", "both"])
@pytest.mark.parametrize("decompose", [False, True])
def test_pinned_formulas_match_cpu_autograd(dtype, up, decompose):
    if decompose and up != "refl":
        pytest.skip("decompose-only has no enhanced output")
    x, illu, e = operands(2, 7, 9, dtype, 3, "cpu")
    e = None if decompose else e
    g_enh, g_refl = upstream(x, 11), upstream(x, 12)
    xs, il, es = x.clone().requires_grad_(), illu.clone().requires_grad_(), None if e is None else e.clone().requires_grad_()
    r, enh = stock(xs, il, es)
    outs = [r] if up == "refl" else [enh] if up == "enh" else [r, enh]
    grads = [g_refl] if up == "refl" else [g_enh] if up == "enh" else [g_refl, g_enh]
    torch.autograd.backward(outs, grads)
    got = M._retinex_grad_ops(x, illu, e, g_refl if up != "enh" else None, g_enh if up != "refl" else None, False,
                              (True, True, e is not None and up != "refl"))
    exact(got[0], xs.grad)
    exact(got[1], il.grad)
    exact(got[2], None if es is None else es.grad)


def test_entry_points_check_their_arguments():
    """Status codes of the two C entries for bad scalars and shapes.  Every pointer is NULL, so no order of the checks can
    reach a launch; the rows that need real pointers are in test_entry_points_null_combinations."""
    import __graft_entry__ as g
    g.ensure_built()
    from retinex_image_enhancement_b200 import native
    L = native.lib()
    fwd, bwd = L.upr_retinex_recombine_maps, L.upr_retinex_recombine_grad
    assert fwd(None, None, None, 3, 0, None, None, 1, 4, 4, 1e-6, None) == -4          # unknown map dtype
    assert fwd(None, None, None, 1, 2, None, None, 1, 4, 4, 1e-6, None) == -4          # unknown flag
    assert fwd(None, None, None, 0, 0, None, None, 1, 0, 4, 1e-6, None) == -2
    assert fwd(None, None, None, 0, 0, None, None, -1, 4, 4, 1e-6, None) == -2
    assert fwd(None, None, None, 2, 1, None, None, 0, 4, 4, 1e-6, None) == 0            # empty batch
    assert fwd(None, None, None, 0, 0, None, None, 1, 4, 4, 1e-6, None) == -1
    assert bwd(None, None, None, 5, 0, None, None, None, None, None, 1, 4, 4, 1e-6, None) == -4
    assert bwd(None, None, None, 0, 4, None, None, None, None, None, 1, 4, 4, 1e-6, None) == -4
    assert bwd(None, None, None, 0, 0, None, None, None, None, None, 1, 4, 0, 1e-6, None) == -2
    assert bwd(None, None, None, 1, 0, None, None, None, None, None, 0, 4, 4, 1e-6, None) == 0   # empty batch
    assert bwd(None, None, None, 0, 0, None, None, None, None, None, 1, 4, 4, 1e-6, None) == -1


def test_cpu_tensors_keep_the_stock_expressions():
    x, illu, e = (t.requires_grad_() for t in operands(1, 4, 4, torch.float32, 1, "cpu"))
    r, enh = M.retinex_recombine(x, illu, e)
    assert type(r.grad_fn).__name__ == "DivBackward0" and type(enh.grad_fn).__name__ == "AddBackward0"
    assert type(M.retinex_decompose(x, illu).grad_fn).__name__ == "DivBackward0"


# ------------------------------------------------------------------------------------------------------------------
# GPU: bit equality with eager autograd on the same device
# ------------------------------------------------------------------------------------------------------------------
SHAPES = [(2, 16, 24, False),     # h*w % 4 == 0: vector kernels
          (3, 7, 9, False),       # h*w % 4 != 0: scalar kernels
          (1, 12, 20, True),      # n = 1, misaligned views: scalar kernels
          (1, 1080, 1920, False)]  # a 1080p frame


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda")


@gpu
@pytest.mark.parametrize("n,h,w,misalign", SHAPES)
@pytest.mark.parametrize("dtype", MAPS)
@pytest.mark.parametrize("autocast", [False, True])
def test_bit_equal_with_eager_autograd(cuda, n, h, w, misalign, dtype, autocast):
    x, illu, e = operands(n, h, w, dtype, n * 100 + h, cuda, misalign)
    for up, x_grad in itertools.product(("enh", "refl", "both"), (False, True)):
        check_case(x, illu, e, x_grad, up, autocast)
    for x_grad in (False, True):   # decompose only
        check_case(x, illu, None, x_grad, "refl", autocast)


@gpu
@pytest.mark.parametrize("dtype", MAPS)
@pytest.mark.parametrize("autocast", [False, True])
@pytest.mark.parametrize("n,h,w,misalign", [(2, 16, 24, False), (3, 7, 9, False)])
def test_edge_values(cuda, dtype, autocast, n, h, w, misalign):
    """GradScaler-sized upstream gradients (x 2^16: fp16 gradients overflow to inf where stock's do), d = 0 from
    illu = -1e-6 (f32 and fp16; in bf16 the sum stays a tiny positive number), NaN in every operand."""
    x, illu, e = operands(n, h, w, dtype, 7, cuda, misalign)
    illu[0, 0, 0, :3] = -1e-6
    x[0, 1, 1, 0] = float("nan")
    illu[-1, 0, 2, 1] = float("nan")
    e[-1, 2, 3, 2] = float("nan")
    x[0, :, 0, 1] = 0.0
    got = check_case(x, illu, e, True, "both", autocast, scale=65536.0)
    if dtype == torch.float16:
        assert torch.isinf(got[4]).any() or torch.isinf(got[3]).any()
    assert torch.isnan(got[2]).any() and (dtype == torch.bfloat16 or torch.isinf(got[0]).any())
    check_case(x, illu, None, True, "refl", autocast, scale=65536.0)


@gpu
def test_forward_keeps_only_its_outputs(cuda):
    """A forward with grad allocates R and enhanced and nothing else (the gradient kernel recomputes what it needs)."""
    x, illu, e = operands(2, 64, 64, torch.float32, 5, cuda)
    x, illu, e = x.requires_grad_(), illu.requires_grad_(), e.requires_grad_()
    growth = {}
    for name, fn in (("fused", M.retinex_recombine), ("stock", stock)):
        torch.cuda.synchronize()
        m0 = torch.cuda.memory_allocated()
        r, enh = fn(x, illu, e)
        torch.cuda.synchronize()
        growth[name] = torch.cuda.memory_allocated() - m0
        del r, enh
    print(f"memory held after the forward, [2,3,64,64] f32: fused {growth['fused']} B, stock {growth['stock']} B")
    assert growth["fused"] == 2 * x.numel() * 4
    assert growth["stock"] > growth["fused"]


@gpu
@pytest.mark.parametrize("dtype", MAPS)
@pytest.mark.parametrize("autocast", [False, True])
def test_create_graph(cuda, dtype, autocast):
    """backward(create_graph=True) evaluates the same formulas as differentiable ops: equal first-order gradients, and a
    second-order gradient close to stock's (fp32 reassociation)."""
    x, illu, e = operands(2, 8, 12, dtype, 9, cuda)
    g_enh, g_refl = upstream(x, 11), upstream(x, 12)
    amp = dtype if dtype != torch.float32 else torch.float16
    res = {}
    for name, fn in (("fused", M.retinex_recombine), ("stock", stock)):
        xs, il, es = x.clone().requires_grad_(), illu.clone().requires_grad_(), e.clone().requires_grad_()
        with torch.autocast("cuda", dtype=amp, enabled=autocast):
            r, enh = fn(xs, il, es)
        grads = torch.autograd.grad([r, enh], [xs, il, es], [g_refl, g_enh], create_graph=True)
        second = torch.autograd.grad(sum(g.float().pow(2).sum() for g in grads), [xs, il, es])
        res[name] = grads, second
    for g, w in zip(res["fused"][0], res["stock"][0]):
        exact(g, w)
    for g, w in zip(res["fused"][1], res["stock"][1]):
        torch.testing.assert_close(g.float(), w.float(), rtol=2e-2 if dtype != torch.float32 else 1e-4, atol=1e-3)


@gpu
def test_entry_points_null_combinations(cuda):
    """Status codes and behaviour of the two C entries for NULL combinations, on real buffers: an output may be left out,
    enhanced needs e, the gradient needs an upstream gradient (and g_enh needs e)."""
    from retinex_image_enhancement_b200 import native
    L = native.lib()
    fwd, bwd = L.upr_retinex_recombine_maps, L.upr_retinex_recombine_grad
    x, illu, e = operands(2, 4, 4, torch.float32, 4, cuda)
    refl, enh = torch.full_like(x, -7.0), torch.full_like(x, -7.0)
    gx, gi, ge = torch.full_like(x, -7.0), torch.full_like(illu, -7.0), torch.full_like(e, -7.0)
    X, I, E, R, N = x.data_ptr(), illu.data_ptr(), e.data_ptr(), refl.data_ptr(), enh.data_ptr()
    s = torch.cuda.current_stream().cuda_stream
    assert fwd(X, I, None, 0, 0, R, N, 2, 4, 4, 1e-6, s) == -1          # enhanced without e
    assert fwd(X, I, E, 0, 0, None, None, 2, 4, 4, 1e-6, s) == -1       # nothing to write
    assert fwd(None, I, E, 0, 0, R, N, 2, 4, 4, 1e-6, s) == -1
    assert fwd(X, None, E, 0, 0, R, N, 2, 4, 4, 1e-6, s) == -1
    assert bwd(X, I, E, 0, 0, None, None, gx.data_ptr(), gi.data_ptr(), ge.data_ptr(), 2, 4, 4, 1e-6, s) == -1
    assert bwd(X, I, None, 0, 0, N, R, gx.data_ptr(), gi.data_ptr(), None, 2, 4, 4, 1e-6, s) == -1   # g_enh without e
    assert bwd(X, I, E, 0, 0, N, R, None, None, None, 2, 4, 4, 1e-6, s) == 0    # no gradient wanted: nothing written
    torch.cuda.synchronize()
    assert (enh == -7.0).all() and (refl == -7.0).all() and (gx == -7.0).all() and (gi == -7.0).all()
    # with e given and enh NULL only R is written
    assert fwd(X, I, E, 0, 0, R, None, 2, 4, 4, 1e-6, s) == 0
    torch.cuda.synchronize()
    exact(refl, stock(x, illu, None)[0])
    assert (enh == -7.0).all()


# ------------------------------------------------------------------------------------------------------------------
# model level
# ------------------------------------------------------------------------------------------------------------------
EAGER_KERNEL = re.compile(r"DivFunctor|div_true|pow", re.I)


def cuda_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]


def captured_maps(monkeypatch):
    """Records (illu, e) of every forward_maps call inside M._forward, with their gradients retained."""
    seen = []
    orig = M._forward_maps

    def spy(m, x):
        illu, e = orig(m, x)
        illu.retain_grad(), e.retain_grad()
        seen.append((illu, e))
        return illu, e

    monkeypatch.setattr(M, "_forward_maps", spy)
    return seen


def loss_of(enh, r):
    return (enh * enh).mean() + (r * 0.25).mean()   # not enh.square(): torch lowers it to a pow kernel


@gpu
def test_up_retinex_trains_through_the_fused_kernels(cuda, monkeypatch):
    torch.manual_seed(0)
    model = M.UP_Retinex().to(cuda).eval()   # eval: BatchNorm statistics fixed, the gradients still flow
    x = torch.rand((1, 3, 64, 64), device=cuda)
    seen = captured_maps(monkeypatch)

    def step():
        enh, r, _illu = model(x)
        loss_of(enh, r).backward()

    names = cuda_kernels(step)
    assert any("k_recombine_vec" in n for n in names) and any("k_recombine_grad_vec" in n for n in names), names
    assert not [n for n in names if EAGER_KERNEL.search(n)]
    # the detector sees the eager arithmetic when it runs
    il2, e2 = (t.detach().requires_grad_() for t in seen[0])
    r2, enh2 = stock(x, il2, e2)
    assert [n for n in cuda_kernels(lambda: loss_of(enh2, r2).backward()) if EAGER_KERNEL.search(n)]

    # boundary gradients equal eager autograd's on the same maps
    seen.clear()
    enh, r, _ = model(x)
    loss_of(enh, r).backward()
    illu, e = seen[-1]
    il_s, e_s = illu.detach().requires_grad_(), e.detach().requires_grad_()
    r_s, enh_s = stock(x, il_s, e_s)
    loss_of(enh_s, r_s).backward()
    exact(r, r_s), exact(enh, enh_s)
    exact(illu.grad, il_s.grad), exact(e.grad, e_s.grad)


class RefLike(nn.Module):
    """A small module with the reference's attribute names and its own stock Retinex arithmetic in forward
    (models/model.py:405-455), as accelerate_reference_model receives it."""

    def __init__(self):
        super().__init__()
        self.ie_net = nn.Sequential(nn.Conv2d(3, 1, 3, padding=1), nn.Sigmoid())
        self.scale1, self.scale2, self.scale3 = (nn.Conv2d(3, 4, 3, padding=1) for _ in range(3))
        self.fusion = nn.Conv2d(12, 4, 1)
        self.output_layer = nn.Conv2d(4, 3, 1)
        self.maps = None

    def retinex_decompose(self, x, illu):
        return x / (illu + 1e-6)

    def multi_scale_enhance(self, x, reflectance, illu):
        full = self.scale1(x)
        parts = [full]
        for branch, s in ((self.scale2, 0.5), (self.scale3, 0.25)):
            y = branch(F.interpolate(x, scale_factor=s, mode="bilinear", align_corners=False))
            parts.append(F.interpolate(y, size=full.shape[2:], mode="bilinear", align_corners=False))
        e = torch.sigmoid(self.output_layer(self.fusion(torch.cat(parts, dim=1))))
        e.retain_grad()
        self.maps = (illu, e)
        return reflectance * e + (1 - reflectance) * (e ** 2)

    def forward(self, x):
        illu = self.ie_net(x)
        illu.retain_grad()
        reflectance = self.retinex_decompose(x, illu)
        return self.multi_scale_enhance(x, reflectance, illu), reflectance, illu


@gpu
def test_accelerated_reference_instance(cuda, monkeypatch):
    torch.manual_seed(1)
    ref = RefLike().to(cuda)
    fast = M.accelerate_reference_model(copy.deepcopy(ref))
    x = torch.rand((2, 3, 32, 48), device=cuda)
    seen = captured_maps(monkeypatch)
    enh, r, _ = fast(x)
    assert type(r.grad_fn).__name__ == "_RetinexFnBackward"
    loss_of(enh, r).backward()
    enh_s, r_s, _ = ref(x)
    loss_of(enh_s, r_s).backward()
    (illu, e), (il_s, e_s) = seen[-1], ref.maps
    exact(illu, il_s), exact(e, e_s), exact(r, r_s), exact(enh, enh_s)
    exact(illu.grad, il_s.grad), exact(e.grad, e_s.grad)
    # decompose alone, through the instance attribute
    il = illu.detach().requires_grad_()
    assert type(fast.retinex_decompose(x, il).grad_fn).__name__ == "_RetinexFnBackward"


@gpu
def test_other_operands_keep_the_stock_expressions(cuda):
    x, illu, e = operands(1, 8, 8, torch.float32, 2, cuda)
    mixed = e.half().requires_grad_()
    r, enh = M.retinex_recombine(x, illu.requires_grad_(), mixed)
    assert type(r.grad_fn).__name__ == "DivBackward0" and type(enh.grad_fn).__name__ == "AddBackward0"
