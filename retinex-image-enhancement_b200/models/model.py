"""Model boundary of the hot path: ``UP_Retinex.forward(x) -> (enhanced, reflectance, illu)``.

What is ON the hot path are the two pointwise Retinex lines around the CNN (reference models/model.py):

    reflectance = x / (illu + 1e-6)                    :405-413  (retinex_decompose)
    enhanced    = R * e + (1 - R) * e**2               :442

Both run in one fused sm_100a kernel (upr_retinex_recombine_f32) at inference (``torch.no_grad()`` / no input requires a
gradient); the enhance drivers go one step further and hand the two CNN outputs ``forward_maps(x) = (illu, e)`` straight to
``native.retinex_clahe`` (recombination fused into the CLAHE histogram kernel).  Under autograd (training) they run as one
``torch.autograd.Function`` on a fused forward and a fused gradient kernel (upr_retinex_recombine_typed / _grad_typed), with
the maps in f32, both in fp16 / bf16, or -- under CUDA autocast, the pair the network emits there -- illu f32 and e fp16 / bf16;
outputs and gradients equal torch autograd through the stock expressions bit for bit.  Other operands (CPU tensors, mixed map
dtypes outside autocast, other shapes) keep the stock expressions.

The CNN itself (illumination U-Net with residual / pre-activation blocks and an optional ASPP bottleneck, three feature-
aggregation branches, :11-403) is dense convolution work that cuDNN already covers and is OUT OF SCOPE for hand-written
kernels (SURVEY.md section 2 row 8).  It is nevertheless built here from stock ``torch.nn`` layers with the reference's module
tree -- same attribute names, same ``nn.Sequential`` positions, hence the same ``state_dict`` keys and shapes -- so that
checkpoints written by the reference trainer (``{'epoch', 'model_state_dict', 'optimizer_state_dict'}``,
trainers/train.py:134-162) load with ``strict=True`` and ``predict`` reproduces the reference for trained weights
(tests/test_host_logic.py::test_model_matches_reference_class).  ``accelerate_reference_model`` does the converse: it takes an
instance of the reference's own class and routes its Retinex arithmetic through the kernels.
"""
from __future__ import annotations

import types

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import native

EPSILON = 1e-6   # models/model.py:411


# ---------------------------------------------------------------------------------------------------
# the two lines on the hot path
# ---------------------------------------------------------------------------------------------------
def _fused_autograd(x: torch.Tensor, illu: torch.Tensor, e=None) -> bool:
    """Whether _RetinexFn takes the operands: CUDA tensors on one device, x [N,3,H,W] f32, illu [N,1,H,W] and e [N,3,H,W]
    (or None) in one map dtype (f32, fp16, bf16) or, while CUDA autocast is enabled, illu f32 and e fp16 / bf16: the maps of
    the network under autocast, whose illumination head adds the f32 mean(x)."""
    if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 4 and x.shape[1] == 3):
        return False
    n, _, h, w = x.shape
    if illu.device != x.device or illu.dtype not in native.MAP_DTYPES or illu.shape != (n, 1, h, w):
        return False
    if e is None:
        return True
    pair = e.dtype == illu.dtype or (illu.dtype == torch.float32 and e.dtype in native.MAP_DTYPES
                                     and torch.is_autocast_enabled("cuda"))
    return pair and e.device == x.device and e.shape == x.shape


def _retinex_grad_ops(x, illu, e, g_refl, g_enh, autocast, need):
    """The gradient kernel's formulas as differentiable torch ops, for backward(create_graph=True): what autograd computes
    through the stock expressions, in its accumulation order (include/upretinex_b200.h, upr_retinex_recombine_grad_typed).
    The illu gradient keeps illu's dtype: f32 (not rounded) for the maps of the network under autocast."""
    with torch.autocast("cuda", enabled=False):
        d = illu + EPSILON
        r = x / d
        g, ge = g_refl, None
        if g_enh is not None:
            ef = e.float() if autocast else e     # autocast evaluates e**2 and its gradient in f32
            t = -(g_enh * (ef * ef))
            g = (t if g_refl is None else t + g_refl) + g_enh * e
            gc = g_enh * (1 - r)
            if not autocast:
                gc = gc.to(e.dtype)
            ge = (g_enh * r).to(e.dtype) + (gc * (2 * ef)).to(e.dtype) if need[2] else None
        gx = g / d if need[0] else None
        gi = (-g * ((x / d) / d)).sum(1, keepdim=True).to(illu.dtype) if need[1] else None
    return gx, gi, ge


class _RetinexFn(torch.autograd.Function):
    """reflectance = x / (illu + 1e-6) and, with e, enhanced = R*e + (1-R)*e**2 on the fused kernels.  Saves only its inputs
    (the gradient kernel recomputes illu + eps, R and e**2) and forms only the gradients that are needed.  Outputs and
    gradients equal torch autograd through the stock expressions, also under CUDA autocast (read at forward time)."""

    @staticmethod
    def forward(ctx, x, illu, e):
        ctx.set_materialize_grads(False)
        ctx.autocast = torch.is_autocast_enabled("cuda")
        refl, enh = native.retinex_recombine_typed(x, illu, e, autocast=ctx.autocast, eps=EPSILON)
        ctx.save_for_backward(x, illu, e)
        return refl if e is None else (refl, enh)

    @staticmethod
    def backward(ctx, g_refl, g_enh=None):
        x, illu, e = ctx.saved_tensors
        if g_refl is None and g_enh is None:
            return None, None, None
        need = (ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.needs_input_grad[2] and g_enh is not None)
        if torch.is_grad_enabled():   # backward(create_graph=True): the gradient must itself be differentiable
            return _retinex_grad_ops(x, illu, e, g_refl, g_enh, ctx.autocast, need)
        return native.retinex_recombine_grad_typed(x, illu, e, g_enh, g_refl, want=need, autocast=ctx.autocast, eps=EPSILON)


def retinex_decompose(x: torch.Tensor, illu: torch.Tensor) -> torch.Tensor:
    """R = x / (illu + 1e-6).  Inference: the sm_100a kernel (CUDA tensors required -- there is no CPU path).  When autograd
    must flow through the line (training): _RetinexFn for the operands it takes, the stock torch expression otherwise."""
    if torch.is_grad_enabled() and (x.requires_grad or illu.requires_grad):
        if _fused_autograd(x, illu):
            return _RetinexFn.apply(x, illu, None)
        return x / (illu + EPSILON)
    if illu.dtype != torch.float32:   # a map from a CNN under autocast
        return native.retinex_recombine_typed(x, illu, None, eps=EPSILON)[0]
    return native.retinex_decompose(x, illu, EPSILON)


def retinex_recombine(x: torch.Tensor, illu: torch.Tensor, enhancement_map: torch.Tensor):
    """(reflectance, enhanced) of models/model.py:412 and :442."""
    needs_grad = torch.is_grad_enabled() and (x.requires_grad or illu.requires_grad or enhancement_map.requires_grad)
    if needs_grad and _fused_autograd(x, illu, enhancement_map):   # training: fused forward + gradient kernels
        return _RetinexFn.apply(x, illu, enhancement_map)
    if needs_grad:   # training on other operands: autograd through the stock torch ops
        reflectance = x / (illu + EPSILON)
        return reflectance, reflectance * enhancement_map + (1 - reflectance) * (enhancement_map ** 2)
    if illu.dtype != torch.float32 or enhancement_map.dtype != torch.float32:   # the maps of a CNN under autocast
        return native.retinex_recombine_typed(x, illu, enhancement_map, autocast=torch.is_autocast_enabled("cuda"), eps=EPSILON)
    return native.retinex_recombine(x, illu, enhancement_map, want_reflectance=True, eps=EPSILON)


def _enhancement_map(m: nn.Module, x: torch.Tensor) -> torch.Tensor:
    """The convolutional part of ``multi_scale_enhance`` (models/model.py:419-440) on any module that owns the reference's
    ``scale1/2/3``, ``fusion`` and ``output_layer``: sigmoid(output_layer(fusion(cat(three scales))))."""
    full = m.scale1(x)
    size = full.shape[2:]
    parts = [full]
    for branch, s in ((m.scale2, 0.5), (m.scale3, 0.25)):
        y = branch(F.interpolate(x, scale_factor=s, mode="bilinear", align_corners=False))
        parts.append(F.interpolate(y, size=size, mode="bilinear", align_corners=False))
    return torch.sigmoid(m.output_layer(m.fusion(torch.cat(parts, dim=1))))


def _forward_maps(m: nn.Module, x: torch.Tensor):
    return m.ie_net(x), _enhancement_map(m, x)


def _forward(m: nn.Module, x: torch.Tensor):
    illu, e = _forward_maps(m, x)
    reflectance, enhanced = retinex_recombine(x.contiguous(), illu.contiguous(), e.contiguous())
    return enhanced, reflectance, illu


# ---------------------------------------------------------------------------------------------------
# stock-torch CNN with the reference's module tree (state_dict compatible)
# ---------------------------------------------------------------------------------------------------
def _conv(cin, cout, k, **kw):
    return nn.Conv2d(cin, cout, kernel_size=k, padding=kw.pop("padding", (k // 2) * kw.get("dilation", 1)), **kw)


def _projection(cin, cout, stride):
    """1x1 projection shortcut where the shape changes, identity (empty Sequential) otherwise."""
    if stride == 1 and cin == cout:
        return nn.Sequential()
    return nn.Sequential(_conv(cin, cout, 1, stride=stride, bias=False), nn.BatchNorm2d(cout))


class EnhancedFAM(nn.Module):
    """Four parallel branches (1x1 | maxpool+1x1 | 3x3,3x3 | 3x3,dilated 3x3) -> 1x1 fusion -> channel gate -> spatial gate
    (models/model.py:11-97)."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        c = out_channels
        self.branch1 = _conv(in_channels, c, 1)
        self.branch2_pool = nn.MaxPool2d(3, stride=1, padding=1)
        self.branch2_conv = _conv(in_channels, c, 1)
        self.branch3_conv1, self.branch3_conv2 = _conv(in_channels, c, 3), _conv(c, c, 3)
        self.branch4_conv1, self.branch4_conv2 = _conv(in_channels, c, 3), _conv(c, c, 3, dilation=2)
        self.fusion = _conv(4 * c, c, 1)
        self.channel_attention = nn.Sequential(nn.AdaptiveAvgPool2d(1), _conv(c, c // 16, 1), nn.ReLU(inplace=True),
                                               _conv(c // 16, c, 1), nn.Sigmoid())
        self.spatial_attention = nn.Sequential(_conv(2, 1, 7), nn.Sigmoid())
        self.relu = nn.ReLU(inplace=True)

    def forward(self, x):
        branches = [self.branch1(x), self.branch2_conv(self.branch2_pool(x)),
                    self.branch3_conv2(self.relu(self.branch3_conv1(x))), self.branch4_conv2(self.relu(self.branch4_conv1(x)))]
        y = self.relu(self.fusion(torch.cat(branches, dim=1)))
        y = y * self.channel_attention(y)
        gate_in = torch.cat([y.mean(dim=1, keepdim=True), y.max(dim=1, keepdim=True)[0]], dim=1)
        return y * self.spatial_attention(gate_in)


class ResBlock(nn.Module):
    """conv-bn-relu-conv-bn + shortcut, relu (models/model.py:100-135)."""

    def __init__(self, in_channels, out_channels, stride=1):
        super().__init__()
        self.conv1 = _conv(in_channels, out_channels, 3, stride=stride, bias=False)
        self.bn1 = nn.BatchNorm2d(out_channels)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = _conv(out_channels, out_channels, 3, bias=False)
        self.bn2 = nn.BatchNorm2d(out_channels)
        self.shortcut = _projection(in_channels, out_channels, stride)

    def forward(self, x):
        y = self.bn2(self.conv2(self.relu(self.bn1(self.conv1(x)))))
        y += self.shortcut(x)
        return self.relu(y)


class PreActResBlock(nn.Module):
    """bn-relu-conv-bn-relu-conv + shortcut taken after the first activation (models/model.py:138-177)."""

    def __init__(self, in_channels, out_channels, stride=1):
        super().__init__()
        self.bn1 = nn.BatchNorm2d(in_channels)
        self.relu = nn.ReLU(inplace=True)
        self.conv1 = _conv(in_channels, out_channels, 3, stride=stride, bias=False)
        self.bn2 = nn.BatchNorm2d(out_channels)
        self.conv2 = _conv(out_channels, out_channels, 3, bias=False)
        self.shortcut = _projection(in_channels, out_channels, stride)

    def forward(self, x):
        a = self.relu(self.bn1(x))
        skip = self.shortcut(a) if len(self.shortcut) > 0 else x
        y = self.conv2(self.relu(self.bn2(self.conv1(a))))
        y += skip
        return y


def _cbr(cin, cout, k, **kw):
    return nn.Sequential(_conv(cin, cout, k, bias=False, **kw), nn.BatchNorm2d(cout), nn.ReLU(inplace=True))


class ASPPModule(nn.Module):
    """1x1 + dilated 3x3 branches + image-level pooling -> 1x1 fusion with dropout (models/model.py:180-249)."""

    def __init__(self, in_channels, out_channels, dilations=(1, 6, 12, 18)):
        super().__init__()
        self.dilations = list(dilations)
        self.conv1x1 = _cbr(in_channels, out_channels, 1)
        self.aspp_branches = nn.ModuleList([_cbr(in_channels, out_channels, 3, dilation=d) for d in self.dilations[1:]])
        self.global_pool = nn.Sequential(nn.AdaptiveAvgPool2d(1), *_cbr(in_channels, out_channels, 1))
        self.fusion = nn.Sequential(*_cbr(out_channels * (len(self.dilations) + 1), out_channels, 1), nn.Dropout(0.1))

    def forward(self, x):
        pooled = F.interpolate(self.global_pool(x), size=x.shape[2:], mode="bilinear", align_corners=False)
        return self.fusion(torch.cat([self.conv1x1(x)] + [b(x) for b in self.aspp_branches] + [pooled], dim=1))


class UpBlock(nn.Module):
    """2x transposed-conv up-sampling + two conv-bn-relu (models/model.py:252-272)."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.up = nn.ConvTranspose2d(in_channels, out_channels, kernel_size=2, stride=2)
        self.conv = nn.Sequential(_conv(out_channels, out_channels, 3), nn.BatchNorm2d(out_channels), nn.ReLU(inplace=True),
                                  _conv(out_channels, out_channels, 3), nn.BatchNorm2d(out_channels), nn.ReLU(inplace=True))

    def forward(self, x):
        return self.conv(self.up(x))


class ResidualIENet(nn.Module):
    """Illumination U-Net: 3 -> 32, three stride-2 encoder blocks to 256 channels, bottleneck (optionally with ASPP), three
    up blocks with additive skips, a residual head added to the channel mean of the input, sigmoid (models/model.py:275-359)."""

    def __init__(self, use_preact=False, use_aspp=False):
        super().__init__()
        self.use_aspp = use_aspp
        block = PreActResBlock if use_preact else ResBlock
        self.input_layer = _conv(3, 32, 3)
        self.enc1, self.enc2, self.enc3 = block(32, 64, stride=2), block(64, 128, stride=2), block(128, 256, stride=2)
        middle = [ASPPModule(256, 256, dilations=[1, 6, 12, 18])] if use_aspp else []
        self.bottleneck = nn.Sequential(block(256, 256), *middle, block(256, 256))
        self.dec3, self.dec2, self.dec1 = UpBlock(256, 128), UpBlock(128, 64), UpBlock(64, 32)
        self.residual_head = nn.Sequential(_conv(32, 32, 3), nn.ReLU(inplace=True), _conv(32, 1, 1))
        self.sigmoid = nn.Sigmoid()

    def forward(self, x):
        s1 = F.relu(self.input_layer(x))
        s2 = self.enc1(s1)
        s3 = self.enc2(s2)
        y = self.bottleneck(self.enc3(s3))
        y = self.dec1(self.dec2(self.dec3(y) + s3) + s2) + s1
        return self.sigmoid(torch.mean(x, dim=1, keepdim=True) + self.residual_head(y))


def _scale_branch(pool):
    head = [nn.MaxPool2d(pool)] if pool > 1 else []
    return nn.Sequential(*head, _conv(3, 32, 3), nn.ReLU(inplace=True), EnhancedFAM(32, 32))


class MultiScaleUP_Retinex(nn.Module):
    """``forward(x) -> (enhanced, reflectance, illu)`` with the reference's module tree (models/model.py:362-455) and the
    Retinex arithmetic on the B200 kernels at inference."""

    def __init__(self, use_preact: bool = True, use_aspp: bool = True):
        super().__init__()
        self.ie_net = ResidualIENet(use_preact=use_preact, use_aspp=use_aspp)
        self.scale1, self.scale2, self.scale3 = _scale_branch(1), _scale_branch(2), _scale_branch(4)
        self.fusion = _conv(96, 32, 1)
        self.output_layer = _conv(32, 3, 1)

    def retinex_decompose(self, x, illu):
        return retinex_decompose(x, illu)

    def enhancement_map(self, x):
        return _enhancement_map(self, x)

    def forward_maps(self, x):
        """The two CNN outputs the Retinex arithmetic consumes: (illumination [B,1,H,W], enhancement map [B,3,H,W]).
        Inference drivers that only need the CLAHE'd result hand them to the fused ``native.retinex_clahe`` instead of
        materialising reflectance and enhanced (``AdaptiveParameterAdjuster.apply_adaptive_enhancement``)."""
        return _forward_maps(self, x)

    def multi_scale_enhance(self, x, reflectance, illu):
        e = _enhancement_map(self, x)
        return reflectance * e + (1 - reflectance) * (e ** 2)

    def forward(self, x):
        return _forward(self, x)


UP_Retinex = MultiScaleUP_Retinex   # same alias as models/model.py:459


def count_parameters(model):
    return sum(p.numel() for p in model.parameters() if p.requires_grad)


def accelerate_reference_model(model: nn.Module) -> nn.Module:
    """Route the Retinex arithmetic of an instance of the REFERENCE class (models/model.py:362-455, real weights / real
    checkpoints) through the kernels: ``retinex_decompose`` and ``forward`` take the fused sm_100a path at inference, and the
    instance gains ``forward_maps(x) -> (illu, enhancement_map)`` -- its own ``ie_net`` plus the convolution / fusion / sigmoid
    part of its ``multi_scale_enhance`` (:419-440) -- which is what ``AdaptiveParameterAdjuster.apply_adaptive_enhancement``
    needs to reach ``upr_retinex_clahe_f32``.  With autograd enabled (training) ``forward`` and ``retinex_decompose`` run the
    fused forward and gradient kernels of ``_RetinexFn``, whose outputs and gradients equal the instance's own stock arithmetic
    bit for bit, also under CUDA autocast, and keep that arithmetic for operands the kernels do not take (CPU tensors, mixed
    map dtypes outside autocast)."""
    for name in ("ie_net", "scale1", "scale2", "scale3", "fusion", "output_layer"):
        if not hasattr(model, name):
            raise TypeError(f"accelerate_reference_model: not a UP_Retinex-like module (no attribute {name!r})")
    model.retinex_decompose = retinex_decompose   # instance attributes shadow the bound methods
    model.forward_maps = types.MethodType(_forward_maps, model)
    model.enhancement_map = types.MethodType(_enhancement_map, model)
    model.forward = types.MethodType(_forward, model)
    return model
