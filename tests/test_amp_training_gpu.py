"""Mixed-precision training through the fused Retinex kernels: the maps the network emits under CUDA autocast, illu f32 and
e fp16 / bf16, through models.model._RetinexFn (upr_retinex_recombine_typed forward, upr_retinex_recombine_grad_typed
gradient).  Outputs and the x / illu / e gradients are compared bit for bit with torch eager autograd through the stock
expressions under the same autocast; the direct typed entry also for the same pairs without autocast."""
import copy
import itertools
import random
import re

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from retinex_image_enhancement_b200.models import model as M

EPS = M.EPSILON
HALF = (torch.float16, torch.bfloat16)
DT = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}
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


def operands(n, h, w, illu_dt, e_dt, seed, device, misalign=False):
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.rand((n, 3, h, w), generator=g)
    illu = (torch.rand((n, 1, h, w), generator=g) * 0.9 + 0.05).to(illu_dt)
    e = torch.rand((n, 3, h, w), generator=g).to(e_dt)
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


def run(fn, x, illu, e, x_grad, up, amp, g_enh, g_refl):
    """Forward through fn(x, illu, e) -> (R, enhanced) under torch.autocast(dtype=amp) (amp None: no autocast), backward from
    the chosen outputs.  -> (R, enhanced, x.grad, illu.grad, e.grad, grad_fn of R)."""
    x = x.detach().clone().requires_grad_(x_grad)
    illu = illu.detach().clone().requires_grad_()
    e = e.detach().clone().requires_grad_()
    with torch.autocast("cuda", dtype=amp or torch.float16, enabled=amp is not None):
        r, enh = fn(x, illu, e)
    outs, grads = [], []
    if up in ("refl", "both"):
        outs.append(r), grads.append(g_refl)
    if up in ("enh", "both"):
        outs.append(enh), grads.append(g_enh)
    torch.autograd.backward(outs, grads)
    return r, enh, x.grad, illu.grad, e.grad, r.grad_fn


def check_case(x, illu, e, x_grad, up, scale=1.0):
    """The fused path under autocast (in e's dtype) against eager autograd through the stock expressions."""
    g_enh, g_refl = upstream(x, 11, scale), upstream(x, 12, scale)
    got = run(M.retinex_recombine, x, illu, e, x_grad, up, e.dtype, g_enh, g_refl)
    want = run(stock, x, illu, e, x_grad, up, e.dtype, g_enh, g_refl)
    assert type(got[5]).__name__ == "_RetinexFnBackward"
    assert got[3].dtype == torch.float32 and (up == "refl" or got[4].dtype == e.dtype)
    for g, w in zip(got[:5], want[:5]):
        exact(g, w)
    return got


# ------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------
def test_typed_grad_entry_checks_its_arguments():
    """Status codes of upr_retinex_recombine_grad_typed for bad pairs, flags and shapes.  Every pointer is NULL, so no order
    of the checks can reach a launch."""
    import __graft_entry__ as g
    g.ensure_built()
    from retinex_image_enhancement_b200 import native
    bwd = native.lib().upr_retinex_recombine_grad_typed

    def call(illu_dt, e_dt, flags, n=1, h=4, w=4):
        return bwd(None, None, illu_dt, None, e_dt, flags, None, None, None, None, None, n, h, w, 1e-6, None)

    for bad in [(0, 3, 0), (0, -1, 0), (3, 1, 0), (-1, 1, 1), (0, 1, 2), (0, 2, 3), (1, 2, 1), (2, 1, 0), (2, 1, 1), (1, 0, 0),
                (2, 0, 1)]:
        assert call(*bad) == -4, bad                        # unknown dtype or flag, (bf16, fp16), 16-bit illu with f32 e
    assert call(0, 1, 1, h=0) == -2 and call(0, 2, 1, w=0) == -2 and call(0, 1, 0, n=-1) == -2
    assert call(0, 3, 0, h=0) == -2                          # the shape is checked first
    for ok in [(0, 0, 0), (0, 0, 1), (0, 1, 0), (0, 1, 1), (0, 2, 0), (0, 2, 1), (1, 1, 1), (2, 2, 0)]:
        assert call(*ok, n=0) == 0, ok                       # empty batch
        assert call(*ok) == -1, ok                           # NULL operands


@pytest.mark.parametrize("e_dt", HALF)
@pytest.mark.parametrize("autocast", [False, True])
@pytest.mark.parametrize("up", ["enh", "refl", "both"])
def test_pinned_formulas_match_cpu_autograd(e_dt, autocast, up):
    """backward(create_graph=True)'s differentiable formulas for (illu f32, e fp16 / bf16) against CPU autograd through the
    stock expressions; autocast's f32 pow is written out as e.float() ** 2."""
    x, illu, e = operands(2, 7, 9, torch.float32, e_dt, 3, "cpu")
    g_enh, g_refl = upstream(x, 11), upstream(x, 12)
    xs, il, es = x.clone().requires_grad_(), illu.clone().requires_grad_(), e.clone().requires_grad_()
    r = xs / (il + EPS)
    enh = r * es + (1 - r) * ((es.float() if autocast else es) ** 2)
    outs = [r] if up == "refl" else [enh] if up == "enh" else [r, enh]
    grads = [g_refl] if up == "refl" else [g_enh] if up == "enh" else [g_refl, g_enh]
    torch.autograd.backward(outs, grads)
    got = M._retinex_grad_ops(x, illu, e, g_refl if up != "enh" else None, g_enh if up != "refl" else None, autocast,
                              (True, True, up != "refl"))
    exact(got[0], xs.grad)
    exact(got[1], il.grad)
    exact(got[2], None if up == "refl" else es.grad)


# ------------------------------------------------------------------------------------------------------------------
# GPU: _RetinexFn under autocast against eager autograd
# ------------------------------------------------------------------------------------------------------------------
SHAPES = [(2, 16, 24, False),     # h*w % 4 == 0: vector kernels
          (3, 7, 9, False),       # h*w % 4 != 0: scalar kernels
          (1, 12, 20, True),      # misaligned views: scalar kernels
          (1, 1080, 1920, False)]  # a 1080p frame


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda")


@gpu
@pytest.mark.parametrize("n,h,w,misalign", SHAPES)
@pytest.mark.parametrize("e_dt", HALF)
def test_bit_equal_with_eager_autograd(cuda, n, h, w, misalign, e_dt):
    x, illu, e = operands(n, h, w, torch.float32, e_dt, n * 100 + h, cuda, misalign)
    for up, x_grad in itertools.product(("enh", "refl", "both"), (False, True)):
        check_case(x, illu, e, x_grad, up)


@gpu
@pytest.mark.parametrize("e_dt", HALF)
@pytest.mark.parametrize("n,h,w,misalign", [(2, 16, 24, False), (3, 7, 9, False)])
def test_edge_values(cuda, e_dt, n, h, w, misalign):
    """GradScaler-sized upstream gradients (x 2^16: fp16 e gradients overflow to inf where stock's do, the f32 illu gradient
    does not), d = 0 from illu = -1e-6 (exact in f32), NaN in every operand."""
    x, illu, e = operands(n, h, w, torch.float32, e_dt, 7, cuda, misalign)
    illu[0, 0, 0, :3] = -1e-6
    x[0, 1, 1, 0] = float("nan")
    illu[-1, 0, 2, 1] = float("nan")
    e[-1, 2, 3, 2] = float("nan")
    x[0, :, 0, 1] = 0.0
    got = check_case(x, illu, e, True, "both", scale=65536.0)
    if e_dt == torch.float16:
        assert torch.isinf(got[4]).any()
    assert torch.isinf(got[0]).any() and torch.isnan(got[2]).any() and torch.isnan(got[3]).any()


@gpu
@pytest.mark.parametrize("e_dt", HALF)
def test_create_graph(cuda, e_dt):
    """backward(create_graph=True) evaluates the same formulas as differentiable ops: equal first-order gradients, and a
    second-order gradient close to stock's (fp32 reassociation)."""
    x, illu, e = operands(2, 8, 12, torch.float32, e_dt, 9, cuda)
    g_enh, g_refl = upstream(x, 11), upstream(x, 12)
    res = {}
    for name, fn in (("fused", M.retinex_recombine), ("stock", stock)):
        xs, il, es = x.clone().requires_grad_(), illu.clone().requires_grad_(), e.clone().requires_grad_()
        with torch.autocast("cuda", dtype=e_dt):
            r, enh = fn(xs, il, es)
        if name == "fused":
            assert type(r.grad_fn).__name__ == "_RetinexFnBackward"
        grads = torch.autograd.grad([r, enh], [xs, il, es], [g_refl, g_enh], create_graph=True)
        second = torch.autograd.grad(sum(g.float().pow(2).sum() for g in grads), [xs, il, es])
        res[name] = grads, second
    for g, w in zip(res["fused"][0], res["stock"][0]):
        exact(g, w)
    for g, w in zip(res["fused"][1], res["stock"][1]):
        torch.testing.assert_close(g.float(), w.float(), rtol=2e-2, atol=1e-3)


@gpu
@pytest.mark.parametrize("illu_dt,e_dt", [(torch.float32, torch.float16), (torch.float32, torch.bfloat16),
                                          (torch.float16, torch.float32), (torch.bfloat16, torch.float16)])
@pytest.mark.parametrize("autocast", [False, True])
def test_other_pairs_keep_the_stock_expressions(cuda, illu_dt, e_dt, autocast):
    """A mixed pair outside autocast, and a pair the kernels do not take, stay on the stock expressions."""
    x, illu, e = operands(1, 8, 8, illu_dt, e_dt, 2, cuda)
    with torch.autocast("cuda", dtype=e_dt if e_dt != torch.float32 else torch.float16, enabled=autocast):
        r, enh = M.retinex_recombine(x, illu.requires_grad_(), e.requires_grad_())
    fused = autocast and illu_dt == torch.float32
    assert type(r.grad_fn).__name__ == ("_RetinexFnBackward" if fused else "DivBackward0")
    assert fused or type(enh.grad_fn).__name__ == "AddBackward0"


# ------------------------------------------------------------------------------------------------------------------
# GPU: the typed gradient entry directly
# ------------------------------------------------------------------------------------------------------------------
def eager_grads(x, illu, e, g_enh, g_refl, amp):
    """R, enhanced and the (x, illu, e) gradients of eager autograd through the stock expressions; amp None = no autocast.
    g_enh None: e receives no gradient."""
    xs, il, es = x.clone().requires_grad_(), illu.clone().requires_grad_(), e.clone().requires_grad_()
    with torch.autocast("cuda", dtype=amp or torch.float16, enabled=amp is not None):
        r, enh = stock(xs, il, es)
    outs = [o for o, g in ((r, g_refl), (enh, g_enh)) if g is not None]
    grads = [g for g in (g_refl, g_enh) if g is not None]
    gx, gi, ge = torch.autograd.grad(outs, [xs, il, es], grads, allow_unused=True)
    return r.detach(), enh.detach(), gx, gi, ge


def amp_of(e_dt, autocast):
    return (e_dt if e_dt != torch.float32 else torch.float16) if autocast else None


@gpu
@pytest.mark.parametrize("e_dt", HALF)
@pytest.mark.parametrize("n,h,w,misalign", [(2, 16, 24, False), (3, 7, 9, False), (1, 12, 20, True)])
def test_mixed_pairs_without_autocast(cuda, e_dt, n, h, w, misalign):
    """flags = 0 with illu f32 and e fp16 / bf16: e**2 and the e-side gradient in e's dtype, as eager autograd without
    autocast evaluates them; the model never produces this pair, the C ABI takes it as upr_retinex_recombine_typed does."""
    from retinex_image_enhancement_b200 import native
    x, illu, e = operands(n, h, w, torch.float32, e_dt, 21 + h, cuda, misalign)
    g_enh, g_refl = upstream(x, 13), upstream(x, 14)
    r, enh, gx, gi, ge = eager_grads(x, illu, e, g_enh, g_refl, None)
    r2, enh2 = native.retinex_recombine_typed(x, illu, e, autocast=False, eps=EPS)
    gx2, gi2, ge2 = native.retinex_recombine_grad_typed(x, illu, e, g_enh, g_refl, autocast=False, eps=EPS)
    for got, want in ((r2, r), (enh2, enh), (gx2, gx), (gi2, gi), (ge2, ge)):
        exact(got, want)


@gpu
def test_typed_entry_null_combinations(cuda):
    """On real buffers: the status codes of the NULL rules, nothing written where a call is refused or nothing is wanted, and
    each gradient alone equal to the same gradient of the full call."""
    from retinex_image_enhancement_b200 import native
    bwd = native.lib().upr_retinex_recombine_grad_typed
    x, illu, e = operands(2, 8, 8, torch.float32, torch.float16, 4, cuda)
    g_enh, g_refl = upstream(x, 15), upstream(x, 16)
    gx, gi, ge = torch.full_like(x, -7.0), torch.full_like(illu, -7.0), torch.full_like(e, -7.0)
    X, I, E, GE, GR = x.data_ptr(), illu.data_ptr(), e.data_ptr(), g_enh.data_ptr(), g_refl.data_ptr()
    s = torch.cuda.current_stream().cuda_stream

    def call(*ptrs, x_=X, i_=I, e_=E):
        return bwd(x_, i_, 0, e_, 1, 1, *ptrs, 2, 8, 8, EPS, s)

    outs = (gx.data_ptr(), gi.data_ptr(), ge.data_ptr())
    assert call(None, None, *outs) == -1                   # no upstream gradient
    assert call(GE, GR, *outs, e_=None) == -1              # g_enh without e
    assert call(None, GR, outs[0], outs[1], outs[2], e_=None) == -1   # g_e without e
    assert call(GE, GR, *outs, x_=None) == -1
    assert call(GE, GR, *outs, i_=None) == -1
    assert call(GE, GR, None, None, None) == 0             # no gradient wanted
    torch.cuda.synchronize()
    assert (gx == -7.0).all() and (gi == -7.0).all() and (ge == -7.0).all()
    full = native.retinex_recombine_grad_typed(x, illu, e, g_enh, g_refl, autocast=True, eps=EPS)
    for k in range(3):
        want = tuple(j == k for j in range(3))
        part = native.retinex_recombine_grad_typed(x, illu, e, g_enh, g_refl, want=want, autocast=True, eps=EPS)
        assert all((p is None) == (not wk) for p, wk in zip(part, want))
        exact(part[k], full[k])
    # decompose only (e NULL): the x and illu gradients of R alone
    gx_r, gi_r, _ = native.retinex_recombine_grad_typed(x, illu, None, None, g_refl, want=(True, True, False), eps=EPS)
    _, _, gx_w, gi_w, _ = eager_grads(x, illu, e, None, g_refl, None)
    exact(gx_r, gx_w), exact(gi_r, gi_w)
    with pytest.raises(TypeError):
        native.retinex_recombine_grad_typed(x, illu.to(torch.bfloat16), e, g_enh, g_refl)


PAIRS = [(torch.float32, torch.float32), (torch.float16, torch.float16), (torch.bfloat16, torch.bfloat16),
         (torch.float32, torch.float16), (torch.float32, torch.bfloat16)]


class Guarded:
    """A tensor of `shape` / `dtype` in the middle of a larger allocation whose margins hold `fill` (NaN for inputs, a
    canary for outputs)."""
    MARGIN = 1024   # elements

    def __init__(self, shape, dtype, fill, offset=0):
        numel = 1
        for s in shape:
            numel *= s
        self.raw = torch.full((2 * self.MARGIN + numel + offset,), fill, dtype=dtype, device="cuda")
        self.lo, self.hi = self.MARGIN + offset, self.MARGIN + offset + numel
        self.t = self.raw[self.lo:self.hi].view(shape)

    def intact(self, fill):
        m = torch.cat([self.raw[:self.lo], self.raw[self.hi:]]).float()
        return bool(torch.isnan(m).all()) if fill != fill else bool((m == fill).all())


@gpu
def test_seeded_sweep_with_guard_bands(cuda):
    """30 random shapes, map pairs, flags, upstream gradients and wanted outputs through the typed entries, inputs between NaN
    margins and outputs between canaries, some misaligned, against eager autograd."""
    from retinex_image_enhancement_b200 import native
    rng = random.Random(20261022)
    canary = -1152.0   # exact in f32, fp16 and bf16
    for case in range(30):
        n, h, w = rng.randint(1, 3), rng.randint(1, 70), rng.randint(1, 70)
        if case % 3 == 0:
            w = 4 * rng.randint(1, 24)   # a whole number of 4-pixel groups: the vector kernels when aligned
        illu_dt, e_dt = rng.choice(PAIRS)
        autocast = rng.random() < 0.6
        up = rng.choice(["enh", "refl", "both"])
        off = rng.choice([0, 0, 1])
        x0, il0, e0 = operands(n, h, w, illu_dt, e_dt, 500 + case, cuda)
        gins = {k: Guarded(t.shape, t.dtype, float("nan"), off) for k, t in (("x", x0), ("illu", il0), ("e", e0))}
        for k, t in (("x", x0), ("illu", il0), ("e", e0)):
            gins[k].t.copy_(t)
        x, illu, e = gins["x"].t, gins["illu"].t, gins["e"].t
        g_enh = upstream(x, case) if up != "refl" else None
        g_refl = upstream(x, case + 1000) if up != "enh" else None
        want = (rng.random() < 0.8, rng.random() < 0.8, up != "refl" and rng.random() < 0.8)
        if not any(want):
            want = (True, False, False)
        outs = [Guarded(x.shape, torch.float32, canary, off), Guarded(illu.shape, illu_dt, canary, off),
                Guarded(e.shape, e_dt, canary, off)]
        refl, enh = Guarded(x.shape, torch.float32, canary, off), Guarded(x.shape, torch.float32, canary, off)
        L = native.lib()
        s = torch.cuda.current_stream().cuda_stream
        flags = int(autocast)
        assert L.upr_retinex_recombine_typed(x.data_ptr(), illu.data_ptr(), DT[illu_dt], e.data_ptr(), DT[e_dt], flags,
                                             refl.t.data_ptr(), enh.t.data_ptr(), n, h, w, EPS, s) == 0
        ptr = [o.t.data_ptr() if wk else None for o, wk in zip(outs, want)]
        assert L.upr_retinex_recombine_grad_typed(x.data_ptr(), illu.data_ptr(), DT[illu_dt], e.data_ptr(), DT[e_dt], flags,
                                                  g_enh.data_ptr() if g_enh is not None else None,
                                                  g_refl.data_ptr() if g_refl is not None else None, *ptr, n, h, w, EPS, s) == 0
        torch.cuda.synchronize()
        r_w, enh_w, *g_w = eager_grads(x, illu, e, g_enh, g_refl, amp_of(e_dt, autocast))
        ctx = f"case {case}: {(n, h, w)} {illu_dt} {e_dt} autocast={autocast} up={up} want={want} off={off}"
        exact(refl.t, r_w), exact(enh.t, enh_w)
        assert refl.intact(canary) and enh.intact(canary), ctx
        for o, wk, gw in zip(outs, want, g_w):
            if wk:
                exact(o.t, gw)
            else:
                assert bool((o.t.float() == canary).all()), ctx
            assert o.intact(canary), ctx
        for k in gins:
            assert gins[k].intact(float("nan")), ctx


# ------------------------------------------------------------------------------------------------------------------
# model level: a training step of UP_Retinex under autocast
# ------------------------------------------------------------------------------------------------------------------
EAGER_KERNEL = re.compile(r"DivFunctor|div_true|pow", re.I)   # the detector of test_retinex_autograd_gpu.py

# Run in a child process: a profiler session leaves process-wide tracing state behind, and later sessions of the suite
# (which look for their own kernels in a trace) must not depend on how many ran before them.
PROFILE_CHILD = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
import torch
from torch.profiler import ProfilerActivity, profile
from retinex_image_enhancement_b200.models import model as M
e_dt = getattr(torch, sys.argv[2])


def kernels(fn):
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]


def loss_of(enh, r):
    return (enh * enh).mean() + (r * 0.25).mean()


torch.manual_seed(0)
model = M.UP_Retinex().cuda().train()
x = torch.rand((2, 3, 64, 64), device="cuda")
maps, orig = [], M._forward_maps
M._forward_maps = lambda m, x: maps.append(orig(m, x)) or maps[-1]


def step():
    with torch.autocast("cuda", dtype=e_dt):
        enh, r, _ = model(x)
        loss = loss_of(enh, r)
    loss.backward()


fused = kernels(step)
il, e = (t.detach().requires_grad_() for t in maps[-1])
with torch.autocast("cuda", dtype=e_dt):
    r = x / (il + M.EPSILON)
    loss = loss_of(r * e + (1 - r) * (e ** 2), r)
stock = kernels(loss.backward)
print(json.dumps({"maps": [str(t.dtype) for t in maps[-1]], "fused": fused, "stock": stock}))
"""


def grad_vec_kernel(e_dt):
    """The demangled or mangled name of k_recombine_grad_vec<float, TE, true>."""
    te, mangled = ("__half", "6__half") if e_dt == torch.float16 else ("__nv_bfloat16", "13__nv_bfloat16")
    return re.compile(rf"k_recombine_grad_vec<float, {te}, true>|k_recombine_grad_vecIf{mangled}Lb1E")


@gpu
@pytest.mark.parametrize("e_dt", HALF)
def test_training_step_runs_the_fused_kernels(cuda, e_dt):
    """A UP_Retinex training step under autocast: forward_maps yields (f32, T), the trace shows the fused forward and the
    (f32, T) gradient kernel and no eager div / pow kernel, and the detector sees the stock lines when they run."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-s", "-c", PROFILE_CHILD, root, str(e_dt).split(".")[1]], capture_output=True,
                       text=True, cwd=root, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["maps"] == ["torch.float32", str(e_dt)]
    names = res["fused"]
    assert any("k_recombine_vec" in n for n in names), names
    assert any(grad_vec_kernel(e_dt).search(n) for n in names), names
    assert not [n for n in names if EAGER_KERNEL.search(n)]
    assert [n for n in res["stock"] if EAGER_KERNEL.search(n)]


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


def params_of(model):
    return {k: p.detach().clone() for k, p in model.named_parameters()}


# Parameter gradients against the stock path.  The backward of the bilinear up-sampling in the enhancement branches
# (upsample_bilinear2d_backward) accumulates with atomics, so torch does not promise the same bits from run to run.  On a B200
# at this size two stock steps agree bit for bit, and the fused step agrees with them exactly; the tolerance below is only for
# a run in which stock itself does not reproduce.
PARAM_RTOL, PARAM_ATOL = 1e-2, 1e-5


@gpu
@pytest.mark.parametrize("e_dt", HALF)
def test_up_retinex_trains_under_autocast(cuda, monkeypatch, e_dt):
    torch.manual_seed(0)
    model = M.UP_Retinex().to(cuda).train()
    x = torch.rand((2, 3, 64, 64), device=cuda)
    seen = captured_maps(monkeypatch)

    # boundary gradients equal eager autograd's on the captured maps
    torch.manual_seed(2)   # dropout in the ASPP bottleneck
    with torch.autocast("cuda", dtype=e_dt):
        enh, r, _ = model(x)
        assert type(r.grad_fn).__name__ == "_RetinexFnBackward"
        loss = loss_of(enh, r)
    loss.backward()
    fused_grads = {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}
    illu, e = seen[-1]
    il_s, e_s = illu.detach().requires_grad_(), e.detach().requires_grad_()
    with torch.autocast("cuda", dtype=e_dt):
        r_s, enh_s = stock(x, il_s, e_s)
        loss_s = loss_of(enh_s, r_s)
    loss_s.backward()
    assert illu.dtype == torch.float32 and e.dtype == e_dt   # forward_maps under autocast: (f32, T)
    exact(r, r_s), exact(enh, enh_s)
    exact(illu.grad, il_s.grad), exact(e.grad, e_s.grad)

    # the same step twice on the stock expressions: the same loss; parameter gradients equal while stock reproduces itself
    monkeypatch.setattr(M, "_fused_autograd", lambda *a: False)
    stock_grads = []
    for _ in range(2):
        model.zero_grad(set_to_none=True)
        torch.manual_seed(2)
        with torch.autocast("cuda", dtype=e_dt):
            enh_k, r_k, _ = model(x)
            assert type(r_k.grad_fn).__name__ == "DivBackward0"
            loss_k = loss_of(enh_k, r_k)
        loss_k.backward()
        exact(loss, loss_k)
        stock_grads.append({k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None})
    assert fused_grads.keys() == stock_grads[0].keys()
    reproducible = all(torch.equal(stock_grads[0][k], stock_grads[1][k]) for k in fused_grads)
    for k, g in fused_grads.items():
        if reproducible:
            exact(g, stock_grads[0][k])
        else:
            torch.testing.assert_close(g, stock_grads[0][k], rtol=PARAM_RTOL, atol=PARAM_ATOL, msg=k)


@gpu
@pytest.mark.parametrize("init_scale", [2.0 ** 16, 2.0 ** 60])
def test_grad_scaler_step(cuda, monkeypatch, init_scale):
    """One fp16 GradScaler step, fused against stock from the same state: the same inf / NaN decision (the scale after
    update()), finite parameters, and parameters left unchanged where the step was skipped."""
    torch.manual_seed(3)
    base = M.UP_Retinex().to(cuda).train()
    x = torch.rand((2, 3, 64, 64), device=cuda)
    result = {}
    for name in ("fused", "stock"):
        model = copy.deepcopy(base)
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)
        scaler = torch.amp.GradScaler("cuda", init_scale=init_scale)
        with monkeypatch.context() as mp:
            if name == "stock":
                mp.setattr(M, "_fused_autograd", lambda *a: False)
            torch.manual_seed(4)
            with torch.autocast("cuda", dtype=torch.float16):
                enh, r, _ = model(x)
                loss = loss_of(enh, r)
            assert (type(r.grad_fn).__name__ == "_RetinexFnBackward") == (name == "fused")
            scaler.scale(loss).backward()
            scaler.step(opt)
            scaler.update()
        result[name] = scaler.get_scale(), params_of(model)
    assert result["fused"][0] == result["stock"][0]
    skipped = result["fused"][0] < init_scale
    assert skipped == (init_scale == 2.0 ** 60)
    before = params_of(base)
    for k, p in result["fused"][1].items():
        assert torch.isfinite(p).all(), k
        if skipped:
            exact(p, before[k])


class RefLike(nn.Module):
    """A small module with the reference's attribute names and its own stock Retinex arithmetic in forward
    (models/model.py:405-455), as accelerate_reference_model receives it.  Its illumination head adds the f32 channel mean of
    x as ResidualIENet's does, so under autocast it emits the same (f32, T) pair."""

    class IENet(nn.Module):
        def __init__(self):
            super().__init__()
            self.conv = nn.Conv2d(3, 1, 3, padding=1)

        def forward(self, x):
            return torch.sigmoid(torch.mean(x, dim=1, keepdim=True) + self.conv(x))

    def __init__(self):
        super().__init__()
        self.ie_net = self.IENet()
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
@pytest.mark.parametrize("e_dt", HALF)
def test_accelerated_reference_instance(cuda, monkeypatch, e_dt):
    torch.manual_seed(5)
    ref = RefLike().to(cuda)
    fast = M.accelerate_reference_model(copy.deepcopy(ref))
    x = torch.rand((2, 3, 32, 48), device=cuda)
    seen = captured_maps(monkeypatch)
    with torch.autocast("cuda", dtype=e_dt):
        enh, r, _ = fast(x)
        loss = loss_of(enh, r)
    assert type(r.grad_fn).__name__ == "_RetinexFnBackward"
    loss.backward()
    with torch.autocast("cuda", dtype=e_dt):
        enh_s, r_s, _ = ref(x)
        loss_s = loss_of(enh_s, r_s)
    loss_s.backward()
    (illu, e), (il_s, e_s) = seen[-1], ref.maps
    assert illu.dtype == torch.float32 and e.dtype == e_dt
    exact(illu, il_s), exact(e, e_s), exact(r, r_s), exact(enh, enh_s)
    exact(illu.grad, il_s.grad), exact(e.grad, e_s.grad)
