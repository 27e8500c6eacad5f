"""Drop-in for the texture-statistics part of the reference's ``losses/loss.py``.

Reference behaviour mirrored (file:line relative to the reference tree):
  * calculate_texture_complexity   losses/loss.py:523-583   ('tv' and 'edge_density', ValueError otherwise)
  * dynamic smoothness weight      losses/loss.py:704-720   clamp(w0 * (1 - 0.8 * mean_B(c)), 0.1, 5.0)

The seven differentiable loss terms (loss.py:12-520) need autograd and stay stock PyTorch: they are out of
scope of the hot path.  ``DynamicSmoothWeight`` is the piece ``TotalLoss.forward`` would call at :707-717;
under data parallelism (one process per GPU, torch.distributed initialised) the batch mean of :710 becomes
ONE all-reduce(SUM) of the two floats [sum of complexity, image count], so every rank derives the same
weight as a single process would on the concatenated batch.
"""
from __future__ import annotations

import torch

from .. import native


def calculate_texture_complexity(img: torch.Tensor, method: str = "tv") -> torch.Tensor:
    """[B,C,H,W] f32 CUDA -> [B] f32 CUDA.  Same error behaviour as the reference for unknown methods."""
    if method not in ("tv", "edge_density"):
        raise ValueError(f"不支持的纹理复杂度计算方法: {method}")
    return native.texture_complexity(img, method)


def batch_texture_stats(img: torch.Tensor, method: str = "tv"):
    """(per-image complexity [B], [sum, B] f32 pair ready for the all-reduce)."""
    if method not in ("tv", "edge_density"):
        raise ValueError(f"不支持的纹理复杂度计算方法: {method}")
    return native.texture_complexity(img, method, want_batch_stats=True)


def all_reduce_batch_stats(stats: torch.Tensor, group=None) -> torch.Tensor:
    """In-place all-reduce(SUM) of the [sum, count] pair when a process group exists; identity otherwise."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    return stats


def weight_from_stats(stats: torch.Tensor, weight_smooth: float = 1.0) -> torch.Tensor:
    """0-dim tensor clamp(w0 * (1 - 0.8 * stats[0]/stats[1]), 0.1, 5.0); CUDA kernel for CUDA stats, and the
    same three fp32 operations in torch for host-side (gloo) tensors."""
    if stats.is_cuda:
        return native.dynamic_smooth_weight(stats, weight_smooth)
    avg = stats[0] / stats[1]
    return torch.clamp(torch.tensor(weight_smooth, dtype=torch.float32) * (1.0 - avg * 0.8), 0.1, 5.0)


class PeerBatchStats:
    """Symmetric-memory exchange buffers for the fused statistics + all-reduce + weight kernel
    (``upr_texture_weight_peer_f32``): one small buffer per rank, mapped into every rank of ``group`` over NVLink
    (``torch.distributed._symmetric_memory``).  Collective: construct it on every rank of the group."""

    def __init__(self, device, group=None):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("PeerBatchStats needs an initialised process group")
        group = dist.group.WORLD if group is None else group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        nfloats = (native.peer_stats_buffer_bytes() + 3) // 4
        self.buf = symm.empty(nfloats, dtype=torch.float32, device=device)
        self.buf.zero_()
        self.handle = symm.rendezvous(self.buf, group=group.group_name)
        self.table = torch.tensor([int(p) for p in self.handle.buffer_ptrs], dtype=torch.int64, device=device)
        torch.cuda.synchronize(device)
        dist.barrier(group=group)          # every buffer is zeroed and mapped before the first exchange
        self.seq = 0

    def next_seq(self) -> int:
        self.seq += 1
        return self.seq

    def check(self) -> None:
        """Raise if an exchange on this rank timed out waiting for a peer (the kernel then returned NaN statistics instead of
        hanging or trapping).  Synchronises the current stream: call it once per epoch / when a NaN weight shows up."""
        call, peer = native.peer_status(self.buf)
        if call != 0:
            raise native.UprError(-4, f"upr_texture_weight_peer_f32: call #{call} on rank {self.rank} timed out waiting for rank "
                                      f"{peer} (every rank must call once per step, in lockstep)")


class DynamicSmoothWeight:
    """``TotalLoss``'s dynamic smoothness weight (losses/loss.py:607-656 constructor arguments
    ``weight_smooth``, ``use_dynamic_smooth_weight``, ``texture_method``).

    ``fused_collective=True`` (data-parallel CUDA training on one NVLink node): statistics, the all-rank batch mean and the
    weight come out of ONE kernel per rank that exchanges the [sum, count] pair through peer memory, instead of a statistics
    kernel + NCCL all-reduce + weight kernel.  Same result on every rank, bit for bit equal to the NCCL path's."""

    def __init__(self, weight_smooth: float = 1.0, use_dynamic_smooth_weight: bool = True, texture_method: str = "tv",
                 group=None, fused_collective: bool = False):
        self.weight_smooth = weight_smooth
        self.use_dynamic_smooth_weight = use_dynamic_smooth_weight
        self.texture_method = texture_method
        self.group = group
        self.fused_collective = fused_collective
        self._peer = None

    def __call__(self, img_low: torch.Tensor) -> torch.Tensor:
        if not self.use_dynamic_smooth_weight:
            return torch.tensor(self.weight_smooth, dtype=torch.float32, device=img_low.device)
        if img_low.is_cuda:
            import torch.distributed as dist
            parallel = dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1
            if parallel and self.fused_collective:
                if self._peer is None:
                    self._peer = PeerBatchStats(img_low.device, self.group)
                p = self._peer
                return native.texture_weight_peer(img_low, self.texture_method, self.weight_smooth, p.table, p.rank, p.world,
                                                  p.next_seq())[2]
            if not parallel:      # one process: nothing to exchange -- statistics + batch mean + weight in ONE kernel
                return native.texture_weight_peer(img_low, self.texture_method, self.weight_smooth, None, 0, 1, 1)[2]
        _per_image, stats = batch_texture_stats(img_low, self.texture_method)
        all_reduce_batch_stats(stats, self.group)
        return weight_from_stats(stats, self.weight_smooth)

    def check_peers(self) -> None:
        """fused_collective only: raise if a peer-memory exchange timed out (see PeerBatchStats.check)."""
        if self._peer is not None:
            self._peer.check()


# ---------------------------------------------------------------------------------------------------
# SURVEY 8f N3: the smoothness term itself (the loss the dynamic weight above multiplies, losses/loss.py:724)
# ---------------------------------------------------------------------------------------------------
class _EdgeSmoothFn(torch.autograd.Function):
    """loss = EdgeAwareSmoothnessLoss(illu_map, img_low); only illu_map carries a gradient.  The kernel that forms the loss
    also writes d loss / d illu (the weights and edge factors are no-grad statistics of img_low), so backward is one scale."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)   # the reference trainer runs the criterion under autocast
    def forward(ctx, illu_map, img_low, lambda_val, alpha):
        need = ctx.needs_input_grad[0]   # (not illu_map.requires_grad: under autocast illu_map is the fp32 copy made by custom_fwd)
        loss3, grad = native.edge_smooth_loss(illu_map.detach(), img_low.detach(), lambda_val, alpha, want_grad=need)
        ctx.save_for_backward(grad if need else torch.empty(0, device=illu_map.device))
        ctx.has_grad = need
        return loss3[0].clone()

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, grad_out):
        (g,) = ctx.saved_tensors
        return (g * grad_out if ctx.has_grad else None), None, None, None


class EdgeAwareSmoothnessLoss(torch.nn.Module):
    """Drop-in for losses/loss.py:61-176 (same constructor arguments, ``forward(illu_map, img_low)`` -> scalar).

    CUDA tensors go through ``upr_edge_smooth_loss_f32`` (forward value and the gradient w.r.t. ``illu_map`` from one pass
    over the batch).  If ``img_low`` itself requires a gradient (it never does in the reference's trainer: it is the input
    image) the stock formulation below runs instead, so autograd still reaches it; CPU tensors raise like every op here."""

    def __init__(self, lambda_val: float = 10.0, alpha: float = 1.0):
        super().__init__()
        self.lambda_val = lambda_val
        self.alpha = alpha

    def forward(self, illu_map: torch.Tensor, img_low: torch.Tensor) -> torch.Tensor:
        if img_low.requires_grad:
            return self._stock(illu_map, img_low)
        return _EdgeSmoothFn.apply(illu_map, img_low, float(self.lambda_val), float(self.alpha))

    def _stock(self, illu_map, img_low):
        # the reference's own sequence of torch ops (losses/loss.py:118-176)
        import torch.nn.functional as F
        gh = lambda t: t[:, :, :, :-1] - t[:, :, :, 1:]      # noqa: E731
        gv = lambda t: t[:, :, :-1, :] - t[:, :, 1:, :]      # noqa: E731
        gray = torch.mean(img_low, dim=1, keepdim=True) if img_low.shape[1] > 1 else img_low
        padded = F.pad(gray, (1, 1, 1, 1), mode="reflect")
        kx = torch.tensor([[-1, 0, 1], [-2, 0, 2], [-1, 0, 1]], dtype=torch.float32, device=img_low.device).view(1, 1, 3, 3)
        ky = torch.tensor([[-1, -2, -1], [0, 0, 0], [1, 2, 1]], dtype=torch.float32, device=img_low.device).view(1, 1, 3, 3)
        edge = torch.sqrt(F.conv2d(padded, kx) ** 2 + F.conv2d(padded, ky) ** 2)
        wh = torch.exp(-self.lambda_val * torch.mean(torch.abs(gh(img_low)), dim=1, keepdim=True))
        wv = torch.exp(-self.lambda_val * torch.mean(torch.abs(gv(img_low)), dim=1, keepdim=True))
        fh = 1 + self.alpha * F.avg_pool2d(edge, kernel_size=(1, wh.shape[3]), stride=1)[:, :, :, :-1]
        fv = 1 + self.alpha * F.avg_pool2d(edge, kernel_size=(wv.shape[2], 1), stride=1)[:, :, :-1, :]
        return torch.mean(wh * fh * torch.abs(gh(illu_map))) + torch.mean(wv * fv * torch.abs(gv(illu_map)))


# ---------------------------------------------------------------------------------------------------
# SURVEY 8f N3: exposure / colour / spatial-consistency losses of the enhanced image from one read of (enhanced, low)
# ---------------------------------------------------------------------------------------------------
class _EnhLossesFn(torch.autograd.Function):
    """(loss_exp, loss_col, loss_spa) = the three statistics losses of losses/loss.py:29-58, :351-368, :404-427.  Only
    ``img_enhanced`` carries a gradient; backward is ONE pass that combines the three upstream gradients."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)   # trainers/train.py:72 calls the criterion under autocast
    def forward(ctx, img_enhanced, img_low, base_target, patch):
        e, l = img_enhanced.detach().contiguous(), img_low.detach().contiguous()
        losses, saved = native.enhanced_image_losses(e, l, base_target, patch)
        ctx.save_for_backward(e, l, saved)
        ctx.patch = patch
        return losses[0].clone(), losses[1].clone(), losses[2].clone()

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g_exp, g_col, g_spa):
        e, l, saved = ctx.saved_tensors
        zero = torch.zeros((), dtype=torch.float32, device=e.device)
        up = torch.stack([g if g is not None else zero for g in (g_exp, g_col, g_spa)]).to(torch.float32)
        return native.enhanced_image_losses_grad(e, l, saved, up, ctx.patch), None, None, None


class EnhancedImageLosses:
    """The three modules ``TotalLoss`` calls on the enhanced image (losses/loss.py:672, :674, :675) share one evaluation: the
    first of ``exposure`` / ``color`` / ``spatial`` that sees a new ``img_enhanced`` runs the fused kernels, the other two
    read the same result.  The cache is keyed on the two tensor objects, their version counters AND whether autograd records
    the evaluation (a value computed under ``torch.no_grad()`` must not be handed to a later grad-enabled call on the same
    tensor); it is dropped as soon as all three terms have been served, so that it never pins the previous iteration's tensors
    and autograd graph."""

    def __init__(self, patch_size: int = 16, base_target_exposure: float = 0.6):
        self.patch_size, self.base_target_exposure = patch_size, base_target_exposure
        self.clear()

    def evaluate(self, img_enhanced, img_low=None, index=None):
        # the cache keeps the two tensor OBJECTS alive and compares by identity + version counter (an id() alone could be
        # re-used by the next iteration's tensor once this one is freed)
        same_enh = self._enh is img_enhanced
        if img_low is None:
            img_low = self._low if (same_enh and self._low is not None) else img_enhanced
        key = (img_enhanced._version, img_low._version, bool(torch.is_grad_enabled() and img_enhanced.requires_grad))
        hit = same_enh and self._low is img_low and self._versions == key
        if not hit:
            self._val = _EnhLossesFn.apply(img_enhanced, img_low, float(self.base_target_exposure), int(self.patch_size))
            self._enh, self._low, self._versions, self._served = img_enhanced, img_low, key, set()
        val = self._val
        if index is not None:
            self._served.add(index)
            if len(self._served) == 3:
                self.clear()
        return val

    def clear(self):
        """Drop the cached evaluation (and the references to its tensors and autograd graph)."""
        self._enh, self._low, self._versions, self._val, self._served = None, None, None, None, set()

    class _Term(torch.nn.Module):
        def __init__(self, owner, index, takes_low):
            super().__init__()
            self._owner, self._index, self._takes_low = [owner], index, takes_low   # list: keep the owner out of nn.Module's registry

        def forward(self, img_enhanced, img_low=None):
            return self._owner[0].evaluate(img_enhanced, img_low, self._index)[self._index]

    def exposure(self):
        """Drop-in for AdaptiveExposureLoss: forward(img_enhanced, img_low)."""
        return self._Term(self, 0, True)

    def color(self):
        """Drop-in for ColorLoss: forward(img_enhanced) -- reuses the evaluation of the same tensor (TotalLoss calls the
        exposure term first, loss.py:672-674); called on its own it pairs the image with itself, which the colour term ignores."""
        return self._Term(self, 1, False)

    def spatial(self):
        """Drop-in for SpatialConsistencyLoss: forward(img_enhanced, img_low)."""
        return self._Term(self, 2, True)


# ---------------------------------------------------------------------------------------------------
# The reference's TotalLoss (losses/loss.py:607-760) with the hot-path pieces swapped in
# ---------------------------------------------------------------------------------------------------
def accelerate_reference_total_loss(total_loss, group=None):
    """Route the pieces of an instance of the REFERENCE ``TotalLoss`` that this package implements through the kernels, in
    place, and return it.  The constructor, ``forward(img_low, img_enhanced, illu_map, reflectance=None, epoch=0)`` and the
    ``(total, dict)`` result stay the reference's own:

      * ``smoothness_loss`` (losses/loss.py:623, called at :673) becomes ``EdgeAwareSmoothnessLoss`` above with the same
        ``lambda_val`` / ``alpha`` (loss and gradient from ``upr_edge_smooth_loss_f32``);
      * ``exposure_loss``, ``color_loss`` and ``spatial_loss`` (:622-625, called at :672-675) become the three views of ONE
        fused evaluation (``EnhancedImageLosses``: ``upr_enh_losses_f32`` forward, ``upr_enh_losses_grad_f32`` backward);
      * ``calculate_texture_complexity`` as seen by ``TotalLoss.forward`` (:707) becomes the kernel version; under data
        parallelism (torch.distributed initialised, world > 1) it returns the ALL-RANK batch mean in every element, so that
        ``torch.mean`` at :710 -- and hence the weight of :716-717 -- is the single-process value on every rank (one
        all-reduce of two floats).

    The remaining terms (decoupling, perceptual, frequency) are the reference's own modules."""
    import sys

    old = total_loss.smoothness_loss
    total_loss.smoothness_loss = EdgeAwareSmoothnessLoss(getattr(old, "lambda_val", 10.0), getattr(old, "alpha", 1.0))
    if all(hasattr(total_loss, a) for a in ("exposure_loss", "color_loss", "spatial_loss")):
        ex = total_loss.exposure_loss
        fused = EnhancedImageLosses(getattr(ex, "patch_size", 16), getattr(ex, "base_target_exposure", 0.6))
        total_loss.exposure_loss, total_loss.color_loss, total_loss.spatial_loss = fused.exposure(), fused.color(), fused.spatial()

    def complexity_for_batch_mean(img, method="tv"):
        per_image, stats = batch_texture_stats(img, method)
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            all_reduce_batch_stats(stats, group)
            return (stats[0] / stats[1]).expand(per_image.shape[0])
        return per_image

    mod = sys.modules.get(type(total_loss).__module__)
    if mod is not None and hasattr(mod, "calculate_texture_complexity"):
        mod.calculate_texture_complexity = complexity_for_batch_mean
    total_loss._upr_complexity = complexity_for_batch_mean
    return total_loss
