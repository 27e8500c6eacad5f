"""Argument checks of the native wrappers: a tensor that does not fit what the entry point will read or write raises in Python,
before anything is launched.  A refused `out` lives in a canary-filled allocation that must come back untouched, which shows
that no kernel ran.  The in-place calls the wrappers have always accepted keep working."""
import pytest
import torch

pytestmark = pytest.mark.gpu
N, H, W = 2, 64, 96
SHAPE = (N, 3, H, W)
NUMEL = N * 3 * H * W
PAD = 1 << 14
CANARY = 77.0      # outside [0, 1], where every one of these kernels writes


@pytest.fixture(scope="module")
def native():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from retinex_image_enhancement_b200 import native as nat
    assert nat.lib().upr_device_check() == 0
    return nat


@pytest.fixture(scope="module")
def data():
    g = torch.Generator(device="cuda").manual_seed(3)
    return torch.rand(SHAPE, device="cuda", generator=g), torch.rand(SHAPE, device="cuda", generator=g) * 1.2


def bad_out(kind):
    """(slab, out): a canary-filled allocation and an `out` inside it that does not fit [N,3,H,W] f32.  A launch would write
    NUMEL floats from out.data_ptr() on, which stay inside the slab and change it."""
    slab = torch.full((2 * NUMEL + PAD,), CANARY, dtype=torch.float16 if kind == "wrong_dtype" else torch.float32, device="cuda")
    if kind == "wrong_dtype":
        return slab, slab[:NUMEL].view(SHAPE)
    if kind == "undersized":
        return slab, slab[:NUMEL - NUMEL // N].view(N - 1, 3, H, W)
    return slab, slab[:2 * NUMEL].view(N, 3, H, 2 * W)[..., ::2]      # non-contiguous


OUT_CALLS = {
    "scale_clamp": lambda nat, x, enh, out: nat.scale_clamp(enh, torch.ones(N, device="cuda"), out=out),
    "attention_apply": lambda nat, x, enh, out: nat.attention_apply(enh, nat.attention(x), out=out),
    "content_aware_apply": lambda nat, x, enh, out: nat.content_aware_apply(x, enh, out=out),
    "content_multiscale_apply": lambda nat, x, enh, out: nat.content_multiscale_apply(x, enh, out=out),
    "content_multiscale_apply_gain": lambda nat, x, enh, out: nat.content_multiscale_apply(x, enh, out=out,
                                                                                           gain=torch.ones(N, device="cuda")),
}


@pytest.mark.parametrize("kind", ["undersized", "wrong_dtype", "non_contiguous"])
@pytest.mark.parametrize("op", sorted(OUT_CALLS))
def test_bad_out_is_refused_before_launch(native, data, op, kind):
    slab, out = bad_out(kind)
    with pytest.raises(ValueError):
        OUT_CALLS[op](native, *data, out)
    torch.cuda.synchronize()
    assert bool((slab == CANARY).all())


IN_PLACE = {   # op -> (what the tensor t starts as, the call that reads t and writes `out`)
    "clahe_lab": ("x", lambda nat, x, t, out: nat.clahe_lab(t, out=out)),
    "clahe_lab_u8": ("x8", lambda nat, x, t, out: nat.clahe_lab_u8(t, out=out)),
    "multiscale_enhance": ("enh", lambda nat, x, t, out: nat.multiscale_enhance(x, t, out=out)[0]),
    "scale_clamp": ("enh", lambda nat, x, t, out: nat.scale_clamp(t, torch.linspace(0.5, 1.5, N, device="cuda"), out=out)),
    "content_aware_apply": ("enh", lambda nat, x, t, out: nat.content_aware_apply(x, t, out=out)),
}


@pytest.mark.parametrize("op", sorted(IN_PLACE))
def test_in_place_calls_match_out_of_place(native, data, op):
    x, enh = data
    src, call = IN_PLACE[op]
    t = {"x": x, "enh": enh, "x8": (x * 255).to(torch.uint8).permute(0, 2, 3, 1)}[src].contiguous().clone()
    ref = call(native, x, t, None)
    got = call(native, x, t, t)
    assert got.data_ptr() == t.data_ptr() and torch.equal(got, ref)


@pytest.fixture(scope="module")
def losses_args(native, data):
    enh, low = data[1][:, :, :32, :48].contiguous(), data[0][:, :, :32, :48].contiguous()
    _losses, saved = native.enhanced_image_losses(enh, low)
    return enh, low, saved, torch.ones(3, device="cuda")


@pytest.mark.parametrize("case", ["one_channel_enhanced", "img_low_shape", "short_saved", "short_upstream3"])
def test_losses_grad_checks_every_size(native, losses_args, case):
    enh, low, saved, up = losses_args
    native.enhanced_image_losses_grad(enh, low, saved, up)
    args = {"one_channel_enhanced": (enh[:, :1].contiguous(), low, saved, up), "img_low_shape": (enh, low[:1], saved, up),
            "short_saved": (enh, low, saved[:-1], up), "short_upstream3": (enh, low, saved, up[:2])}[case]
    with pytest.raises(ValueError):
        native.enhanced_image_losses_grad(*args)


def test_dynamic_smooth_weight_needs_the_pair(native):
    with pytest.raises(ValueError):
        native.dynamic_smooth_weight(torch.ones(1, device="cuda"))


@pytest.mark.parametrize("case,exc", [("int32", TypeError), ("host", RuntimeError), ("short", ValueError)])
def test_texture_weight_peer_checks_the_table(native, data, case, exc):
    # every table still holds the address of a real exchange buffer, so that a call which got through would run a valid
    # single-rank exchange; an untouched (all-zero) buffer shows that it did not
    buf = torch.zeros((native.peer_stats_buffer_bytes() + 3) // 4, device="cuda")
    full = torch.tensor([buf.data_ptr()], dtype=torch.int64, device="cuda")
    table = {"int32": full.view(torch.int32), "host": full.cpu().pin_memory(), "short": full[:0]}[case]
    with pytest.raises(exc):
        native.texture_weight_peer(data[0], "tv", 1.0, table, 0, 1, 1)
    torch.cuda.synchronize()
    assert not bool(buf.any())


def test_mixed_devices_are_refused(native, data):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    x, enh = data
    slab = torch.full((NUMEL + PAD,), CANARY, device=x.device)
    with pytest.raises(ValueError):
        native.content_aware_apply(x, enh.to("cuda:1"), out=slab[:NUMEL].view(SHAPE))
    with pytest.raises(ValueError):
        native.scale_clamp(enh, torch.ones(N, device="cuda:1"), out=slab[:NUMEL].view(SHAPE))
    torch.cuda.synchronize(x.device)
    assert bool((slab == CANARY).all())
