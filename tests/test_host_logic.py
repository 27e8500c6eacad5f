"""CPU-only checks of the host-side logic: histogram features, sharding, letterbox boundary, CLI flags, the model
contract and the world_size-2 data-parallel batch statistics (gloo)."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import oracle as O


def test_features_from_histogram_match_oracle():
    from retinex_image_enhancement_b200.enhancers._stats import features_from_histogram
    x = O.kat_input(2, 400, 600, "dark")
    h = O.brightness_hist(x)
    got = features_from_histogram(h.astype(np.int64))[0]
    ref = O.features_from_hist(h)
    assert got == ref


def test_adjust_rules_match_oracle(golden):
    from retinex_image_enhancement_b200.enhancers._stats import features_from_histogram
    from retinex_image_enhancement_b200.enhancers.adaptive_params import AdaptiveParameterAdjuster
    adj = AdaptiveParameterAdjuster()
    for rec in golden["bright"]:
        x = O.kat_input(rec["seed"], rec["h"], rec["w"], rec["kind"])
        f = features_from_histogram(O.brightness_hist(x).astype(np.int64))[0]
        assert adj._rules(f) == rec["params"]


@pytest.mark.parametrize("n,world", [(10, 4), (3, 8), (64, 8), (0, 2), (7, 1)])
def test_shard_for_rank_partitions(n, world):
    from retinex_image_enhancement_b200.enhancers.simple_enhance import shard_for_rank
    items = list(range(n))
    parts = [shard_for_rank(items, r, world) for r in range(world)]
    assert sum(parts, []) == items                       # contiguous blocks, every frame exactly once
    assert max(map(len, parts)) - min(map(len, parts)) <= 1


def test_letterbox_identity_and_resize():
    cv2 = pytest.importorskip("cv2")
    from retinex_image_enhancement_b200.utils.letterbox import letterbox_tensor
    rng = np.random.default_rng(3)
    u8 = rng.integers(0, 256, (3, 50, 70), dtype=np.uint8)
    t = torch.from_numpy(u8.astype(np.float32) / 255.0)
    same, ratio, pad = letterbox_tensor(t, new_shape=(50, 70), auto=True, scaleup=False)
    assert torch.equal(same, t) and ratio == (1.0, 1.0) and pad == (0.0, 0.0)
    small, ratio, pad = letterbox_tensor(t, new_shape=32, auto=True, scaleup=False)
    r = min(32 / 50, 32 / 70)
    unpad = (int(round(70 * r)), int(round(50 * r)))
    ref = cv2.resize(u8.transpose(1, 2, 0), unpad, interpolation=cv2.INTER_LINEAR)
    dh = ((32 - unpad[1]) % 32) / 2
    ref = cv2.copyMakeBorder(ref, int(round(dh - 0.1)), int(round(dh + 0.1)), 0, 0, cv2.BORDER_CONSTANT, value=(114, 114, 114))
    assert np.array_equal((small.numpy().transpose(1, 2, 0) * 255).round().astype(np.uint8), ref)


def test_cli_flags_of_the_reference_are_accepted():
    from retinex_image_enhancement_b200.cli import build_main_parser
    a, unknown = build_main_parser().parse_known_args(
        ["--mode", "enhance", "--input_path", "d", "--output_dir", "o", "--max_size", "512", "--device", "cuda", "--multi_scale",
         "--content_aware", "--use_preact", "--use_aspp", "--batch_size", "8"])
    assert a.mode == "enhance" and a.multi_scale and a.content_aware and a.max_size == 512 and unknown == ["--batch_size", "8"]


def test_rank_to_gpu_binding_logic(monkeypatch):
    """cli._device / resolve_device under torchrun: rank r of a node works on cuda:LOCAL_RANK (CPU container: torch.cuda is
    faked; the real two-GPU check is tests/test_drivers_gpu.py::test_ranks_bind_to_their_own_gpu)."""
    from retinex_image_enhancement_b200 import cli, native
    from retinex_image_enhancement_b200.enhancers import simple_enhance as S
    calls = []
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "device_count", lambda: 8)
    monkeypatch.setattr(torch.cuda, "set_device", lambda d: calls.append(d))
    monkeypatch.setattr(torch.cuda, "current_device", lambda: 0)
    monkeypatch.setattr(native, "bind_to_gpu_numa_node", lambda d: True)
    for rank in (0, 5):
        monkeypatch.setenv("WORLD_SIZE", "8")
        monkeypatch.setenv("LOCAL_RANK", str(rank))
        assert cli._device(None) == f"cuda:{rank}" and S.resolve_device("cuda") == f"cuda:{rank}"
        assert calls[-1] == rank
    assert S.resolve_device("cuda:3") == "cuda:3" and S.resolve_device("cpu") == "cpu"
    monkeypatch.delenv("WORLD_SIZE")
    monkeypatch.delenv("LOCAL_RANK")
    assert S.resolve_device(None) == "cuda:0"


def test_cli_defaults_are_the_references(tmp_path, capsys):
    """main.py:29-44: --mode predict, --input_path ./data/test, --checkpoint ./checkpoints/best_model.pth; predict mode without
    the checkpoint file prints the reference's message and does nothing (main.py:152-157)."""
    from retinex_image_enhancement_b200 import cli
    a = cli.build_main_parser().parse_args([])
    assert (a.mode, a.input_path, a.checkpoint, a.output_dir) == ("predict", "./data/test", "./checkpoints/best_model.pth", "./results")
    assert cli.main(["--checkpoint", str(tmp_path / "nope.pth"), "--output_dir", str(tmp_path / "o")]) == 1
    assert "找不到模型检查点文件" in capsys.readouterr().out and not (tmp_path / "o").exists()
    with pytest.raises(SystemExit):
        cli.main(["--mode", "enhance", "--input_path", str(tmp_path / "missing_dir")])


def test_enh_losses_cache_is_keyed_on_grad_mode_and_released(monkeypatch):
    """EnhancedImageLosses: an evaluation made under no_grad is not handed to a grad-enabled call on the same tensor, and the
    cache lets go of its tensors once the three terms have been served (kernels faked: CPU container)."""
    from retinex_image_enhancement_b200.losses import loss as L
    n_eval = []

    class FakeFn:
        @staticmethod
        def apply(e, l, base, patch):
            n_eval.append(torch.is_grad_enabled())
            v = e.sum() * 0 + len(n_eval)
            return v, v, v
    monkeypatch.setattr(L, "_EnhLossesFn", FakeFn)
    fused = L.EnhancedImageLosses()
    t_exp, t_col, t_spa = fused.exposure(), fused.color(), fused.spatial()
    e, low = torch.rand(1, 3, 8, 8, requires_grad=True), torch.rand(1, 3, 8, 8)
    with torch.no_grad():
        a = t_exp(e, low)
    b = t_exp(e, low)                       # grad mode changed -> new evaluation
    assert n_eval == [False, True] and a.item() == 1.0 and b.detach().item() == 2.0
    assert t_col(e).detach().item() == 2.0 and t_spa(e, low).detach().item() == 2.0 and len(n_eval) == 2    # shared
    assert fused._enh is None and fused._val is None          # all three served -> released


def test_model_contract_training_path_on_cpu():
    from retinex_image_enhancement_b200.models.model import UP_Retinex, retinex_recombine
    m = UP_Retinex(use_preact=False, use_aspp=False)
    x = torch.rand(2, 3, 32, 48)
    enhanced, reflectance, illu = m(x)                      # autograd enabled: stock torch ops
    assert enhanced.shape == x.shape and reflectance.shape == x.shape and illu.shape == (2, 1, 32, 48)
    enhanced.mean().backward()
    assert m.output_layer.weight.grad is not None
    with torch.no_grad(), pytest.raises(RuntimeError):      # inference needs the CUDA kernel: no CPU path
        retinex_recombine(x, illu.detach(), x)


def test_hot_path_ops_refuse_cpu_tensors():
    from retinex_image_enhancement_b200 import native
    x = torch.rand(1, 3, 16, 16)
    for fn in (native.clahe_lab, native.brightness_hist, native.multiscale_stats, native.saliency, native.attention,
               native.texture_complexity):
        with pytest.raises(RuntimeError):
            fn(x)
    with pytest.raises(RuntimeError):
        native.clahe_lab_u8(torch.zeros((1, 16, 16, 3), dtype=torch.uint8))
    with pytest.raises(RuntimeError):
        native.clahe_lab_f32_u8(x)
    with pytest.raises(RuntimeError):
        native.edge_smooth_loss(torch.rand(1, 1, 16, 16), x)
    from retinex_image_enhancement_b200.losses.loss import EdgeAwareSmoothnessLoss, EnhancedImageLosses
    with pytest.raises(RuntimeError):
        EdgeAwareSmoothnessLoss()(torch.rand(1, 1, 16, 16), x)
    with pytest.raises(RuntimeError):
        native.enhanced_image_losses(x, x)
    with pytest.raises(RuntimeError):
        EnhancedImageLosses().exposure()(x, x)


# ---- world_size 2 over gloo: the batch statistics of the dynamic smoothness weight -------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _dp_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    from oracle import oracle as Or
    from retinex_image_enhancement_b200.enhancers.simple_enhance import shard_for_rank
    from retinex_image_enhancement_b200.losses.loss import all_reduce_batch_stats, weight_from_stats
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    full = np.random.default_rng(11).random((8, 3, 64, 64), dtype=np.float32)
    mine = shard_for_rank(list(range(8)))                       # env-driven sharding
    local = Or.texture_tv(full[mine])                             # stand-in for the per-rank CUDA kernel
    stats = torch.tensor([np.float32(local.sum(dtype=np.float32)), float(len(mine))], dtype=torch.float32)
    all_reduce_batch_stats(stats)
    w = weight_from_stats(stats, 1.0)
    np.save(os.path.join(out_dir, f"w{rank}.npy"), np.array([float(w), float(stats[0]), float(stats[1])]))
    dist.destroy_process_group()


def test_dp_batch_stats_world2_gloo(tmp_path):
    import torch.multiprocessing as mp
    port = _free_port()
    mp.spawn(_dp_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    full = np.random.default_rng(11).random((8, 3, 64, 64), dtype=np.float32)
    ref = O.dynamic_smooth_weight(O.texture_tv(full))
    r0, r1 = np.load(tmp_path / "w0.npy"), np.load(tmp_path / "w1.npy")
    assert np.array_equal(r0, r1)                                # every rank derives the same weight
    assert r0[2] == 8.0 and abs(r0[0] - ref) <= 1e-6


def test_accelerate_reference_total_loss_patches_the_real_class(monkeypatch):
    """With the unmodified reference at hand (UPR_REFERENCE): the names accelerate_reference_total_loss relies on exist in
    the unmodified losses/loss.py -- TotalLoss().smoothness_loss and the module-level calculate_texture_complexity."""
    ref = os.environ.get("UPR_REFERENCE", "")
    if not os.path.isdir(os.path.join(ref, "losses")):
        pytest.skip("set UPR_REFERENCE to an unmodified checkout of xh92117/Retinex-image-Enhancement to run this comparison")
    import importlib.util
    import sys
    import types
    monkeypatch.setitem(sys.modules, "matplotlib", types.ModuleType("matplotlib"))
    spec = importlib.util.spec_from_file_location("upr_ref_losses", os.path.join(ref, "losses", "loss.py"))
    mod = importlib.util.module_from_spec(spec)
    monkeypatch.setitem(sys.modules, "upr_ref_losses", mod)
    spec.loader.exec_module(mod)
    monkeypatch.setattr(mod, "PerceptualLoss", lambda *a, **k: torch.nn.Identity())      # the real one downloads VGG19
    total = mod.TotalLoss()
    lam, alpha = total.smoothness_loss.lambda_val, total.smoothness_loss.alpha
    from retinex_image_enhancement_b200.losses import loss as L
    out = L.accelerate_reference_total_loss(total)
    assert out is total and isinstance(total.smoothness_loss, L.EdgeAwareSmoothnessLoss)
    assert (total.smoothness_loss.lambda_val, total.smoothness_loss.alpha) == (lam, alpha)
    assert mod.calculate_texture_complexity is total._upr_complexity
    # the three statistics losses of the enhanced image are views of one fused evaluation
    assert type(total.exposure_loss).__name__ == type(total.color_loss).__name__ == type(total.spatial_loss).__name__ == "_Term"
    assert total.exposure_loss._owner[0] is total.color_loss._owner[0] is total.spatial_loss._owner[0]
    assert (total.exposure_loss._owner[0].patch_size, total.exposure_loss._owner[0].base_target_exposure) == (16, 0.6)


def _reference_model_module(monkeypatch):
    ref = os.environ.get("UPR_REFERENCE", "")
    if not os.path.isfile(os.path.join(ref, "models", "model.py")):
        pytest.skip("set UPR_REFERENCE to an unmodified checkout of xh92117/Retinex-image-Enhancement to run this comparison")
    import importlib.util
    import sys
    spec = importlib.util.spec_from_file_location("upr_ref_model", os.path.join(ref, "models", "model.py"))
    mod = importlib.util.module_from_spec(spec)
    monkeypatch.setitem(sys.modules, "upr_ref_model", mod)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("use_preact,use_aspp", [(False, False), (True, True)])
def test_model_matches_reference_class(monkeypatch, use_preact, use_aspp):
    """With the unmodified reference at hand (UPR_REFERENCE): this package's UP_Retinex has the reference's module tree -- a state_dict of the unmodified class
    loads with strict=True (the trainer's checkpoint format, trainers/train.py:134-162) and the forward pass reproduces the
    reference's three outputs bit for bit (stock torch ops on both sides: CPU, autograd enabled)."""
    mod = _reference_model_module(monkeypatch)
    from retinex_image_enhancement_b200.models.model import UP_Retinex, count_parameters
    torch.manual_seed(5)
    theirs = mod.UP_Retinex(use_preact=use_preact, use_aspp=use_aspp).eval()
    for m in theirs.modules():                      # non-trivial batch-norm statistics
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.uniform_(-0.2, 0.2); m.running_var.uniform_(0.5, 1.5)
    ours = UP_Retinex(use_preact=use_preact, use_aspp=use_aspp).eval()
    sd = theirs.state_dict()
    assert list(ours.state_dict().keys()) == list(sd.keys())
    assert all(ours.state_dict()[k].shape == v.shape for k, v in sd.items())
    ours.load_state_dict({"epoch": 3, "model_state_dict": sd}["model_state_dict"], strict=True)
    assert count_parameters(ours) == mod.count_parameters(theirs)
    x = torch.rand(2, 3, 64, 96, requires_grad=True)
    got, want = ours(x), theirs(x)
    for a, b in zip(got, want):
        assert torch.equal(a, b)
    illu, e = ours.forward_maps(x)
    assert torch.equal(illu, want[2]) and e.shape == x.shape


def test_accelerate_reference_model_on_the_real_class(monkeypatch):
    """accelerate_reference_model gives the unmodified reference class forward_maps() (what the fused Retinex + CLAHE entry needs)
    and leaves its autograd behaviour untouched; the recombination of forward_maps' outputs is the class's own `enhanced`."""
    mod = _reference_model_module(monkeypatch)
    from retinex_image_enhancement_b200.models.model import accelerate_reference_model
    torch.manual_seed(6)
    theirs = mod.UP_Retinex(use_preact=False, use_aspp=False).eval()
    x = torch.rand(1, 3, 48, 64, requires_grad=True)
    want = [t.detach().clone() for t in theirs(x)]
    acc = accelerate_reference_model(theirs)
    assert acc is theirs
    got = acc(x)                                    # autograd on: stock ops, same numbers
    for a, b in zip(got, want):
        assert torch.equal(a.detach(), b)
    illu, e = acc.forward_maps(x)
    r = x / (illu + 1e-6)
    assert torch.equal(illu.detach(), want[2]) and torch.equal((r * e + (1 - r) * e ** 2).detach(), want[0])
    with torch.no_grad(), pytest.raises(RuntimeError):   # inference takes the kernel: CUDA tensors only
        acc(x.detach())
    with pytest.raises(TypeError):
        accelerate_reference_model(torch.nn.Linear(2, 2))


def test_bench_dump_outputs_writes_a_fixed_bounded_sample(tmp_path, monkeypatch):
    """bench.py --dump-outputs: small arrays are written whole; a large [N,C,H,W] output becomes the same image rows of every
    frame on every run, float32, within the byte budget."""
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 << 20)
    big = torch.rand((8, 3, 256, 320), generator=torch.Generator().manual_seed(1))
    gain = torch.rand(8, dtype=torch.float64)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"out": big, "gain": gain})
    a, b = np.load(tmp_path / "a" / "out.npy"), np.load(tmp_path / "b" / "out.npy")
    assert a.dtype == np.float32 and np.array_equal(a, b)
    assert a.nbytes <= 2 << 20 and a.shape[:2] == (8, 3) and a.shape[3] == 320 and 1 < a.shape[2] < 256
    src = big.numpy()
    rows = [next(r for r in range(256) if np.array_equal(src[:, :, r], a[:, :, k])) for k in range(a.shape[2])]
    assert rows == sorted(set(rows))
    g = np.load(tmp_path / "a" / "gain.npy")
    assert g.dtype == np.float32 and np.array_equal(g, gain.float().numpy())
    with pytest.raises(ValueError):                     # only [N,C,H,W] outputs can be sampled into the budget
        bench.dump_outputs(str(tmp_path / "c"), {"flat": big.reshape(-1)})
