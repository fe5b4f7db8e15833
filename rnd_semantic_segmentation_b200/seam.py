"""Seam-format producer: make the backbone's last Bottleneck emit the head's fast input format (bf16 channels_last).

    fe = build_feature_extractor(cfg)
    fuse_backbone_tail(fe)        # or install(seam=True) before the trainers / tester build their models

The last Bottleneck of the ResNet backbone (core/models/feature_extractor/resnet.py:106-113) ends with fp32 NCHW passes over
the largest activation of the network: ``bn3`` (a FrozenBatchNorm2d, core/models/layers.py:17-23: ``x * scale + bias``),
``out += identity`` and ``relu``; the head then converts the result to bf16 pixel-major (its feature pack).
``fuse_backbone_tail`` replaces that block's forward by conv1 ... conv3 and ``downsample`` as before, then ONE kernel
(ops.seam_tail) writing ``relu((c * scale + bias) + identity)`` straight as bf16 channels_last, bit-identical to the stock fp32
output converted with ``.to(torch.bfloat16)``.

What changes for the caller:
  - ``feature_extractor(x)`` returns bf16 channels_last (values: the stock features rounded once to bf16);
  - the gradient into the backbone carries that one bf16 rounding (the head's seam-format data gradient is bf16);
  - when one feature map feeds two consumers (FADA: classifier(tgt_fea) and model_D(tgt_fea), aspp_fada.py:91-123), autograd
    sums their gradients in bf16.
The block's ``state_dict()``, ``parameters()`` and class are untouched; ``unfuse_backbone_tail`` restores the original forward.

The kernel is taken only when the block's input is CUDA fp32, conv3's output channels are a multiple of 8 and ``bn3`` is a norm
whose fold is verified: a FrozenBatchNorm2d (buffers only; ``weight * running_var.rsqrt()``, or with ``+ eps`` when the module has
an ``eps``), or an ``nn.BatchNorm2d`` in eval mode whose affine parameters need no gradient in the call.  The fold is checked
against the module's own forward on a small seeded probe the first time and whenever the norm's tensors change (bit-equal for
the frozen norm, within 4 fp32 ulp of the intermediates' magnitude for BatchNorm2d); the fold itself is recomputed from the
norm's current tensors on every call.  Anything else -- a training-mode BatchNorm2d / SyncBatchNorm, another norm, a failed
probe -- runs the block's stock forward.
"""
from __future__ import annotations

import functools
import warnings

import torch
import torch.nn as nn

from . import ops

__all__ = ["fuse_backbone_tail", "unfuse_backbone_tail", "is_fused", "wrap_feature_extractor_factory"]

_BLOCK_ATTRS = ("conv1", "bn1", "conv2", "bn2", "conv3", "bn3", "relu", "downsample")
_FROZEN_BUFFERS = {"weight", "bias", "running_mean", "running_var"}
_PROBE_SHAPE = (2, 3, 5)         # [2, C, 3, 5]


class _FusedForward:
    """What ``fuse_backbone_tail`` installs as the block's instance ``forward``: a plain picklable object (``torch.save`` of a
    whole fused extractor loads again; ``copy.deepcopy`` re-targets it to the copy).  It keeps the forward that was in the
    instance's __dict__ before (normally none) and the key (norm class, eps, data pointers and version counters of the norm's
    tensors) under which the fold last passed or failed its probe."""

    def __init__(self, block, had_forward, old_forward):
        self.block, self.had_forward, self.old_forward = block, had_forward, old_forward
        self.key, self.ok, self.warned = None, False, False

    def __getstate__(self):
        state = dict(self.__dict__)
        state["key"], state["ok"] = None, False            # probe again after loading (other device, other addresses)
        return state

    def __call__(self, x):
        return _fused_forward(self.block, self, x)


def _last_bottleneck(feature_extractor: nn.Module):
    last = None
    for m in feature_extractor.modules():
        if all(hasattr(m, a) for a in _BLOCK_ATTRS):
            last = m
    return last


def _norm_kind(norm):
    """'frozen', 'bn' (eval-mode BatchNorm2d with constant affine parameters in this call) or None (stays stock)."""
    if isinstance(norm, nn.BatchNorm2d):
        if norm.training or norm.running_mean is None or norm.running_var is None:
            return None
        if norm.affine and torch.is_grad_enabled() and (norm.weight.requires_grad or norm.bias.requires_grad):
            return None
        return "bn"
    if isinstance(norm, nn.Module) and not any(True for _ in norm.parameters(recurse=False)):
        bufs = {n for n, b in norm.named_buffers(recurse=False) if b is not None}
        if _FROZEN_BUFFERS <= bufs:
            return "frozen"
    return None


def _norm_tensors(norm, kind):
    if kind == "frozen":
        return [norm.weight, norm.bias, norm.running_mean, norm.running_var]
    return [t for t in (norm.weight, norm.bias, norm.running_mean, norm.running_var) if t is not None]


def _fold(norm, kind):
    """(scale, bias) fp32 [C] such that norm(x) == x * scale + bias."""
    with torch.no_grad():
        if kind == "frozen":
            eps = getattr(norm, "eps", None)
            rv = norm.running_var if eps is None else norm.running_var + eps
            scale = norm.weight * rv.rsqrt()
            bias = norm.bias - norm.running_mean * scale
        else:
            inv = (norm.running_var + norm.eps).rsqrt()
            scale = inv if norm.weight is None else norm.weight * inv
            bias = -norm.running_mean * scale if norm.bias is None else norm.bias - norm.running_mean * scale
        return scale.float().contiguous(), bias.float().contiguous()


def _probe_ok(norm, kind, scale, bias) -> bool:
    """The module's own forward on a seeded [2, C, 3, 5] probe against probe * scale + bias: bit-equal for the frozen norm; for
    BatchNorm2d, whose kernel computes (x - running_mean) * scale + norm.bias instead, within 4 fp32 ulp of
    |probe * scale| + |running_mean * scale| + |bias| elementwise -- the largest intermediates of either form, so the bar holds
    where x - running_mean cancels (measured on a B200: 2-3 ulp of this sum, up to hundreds of ulp of |probe * scale| + |bias|)."""
    C = scale.numel()
    g = torch.Generator().manual_seed(0)
    probe = torch.randn((2, C) + _PROBE_SHAPE[1:], generator=g).to(scale.device)
    with torch.no_grad():
        ref = norm(probe)
        s, b = scale.view(1, C, 1, 1), bias.view(1, C, 1, 1)
        got = probe * s + b
        if not isinstance(ref, torch.Tensor) or ref.shape != got.shape or ref.dtype != torch.float32:
            return False
        if kind == "frozen":
            return bool(torch.equal(ref, got))
        mag = (probe * s).abs() + (norm.running_mean.view(1, C, 1, 1) * s).abs() + b.abs()
        ulp = torch.nextafter(mag, torch.full_like(mag, float("inf"))) - mag
        return bool(((ref - got).abs() <= 4 * ulp).all())


def _folded_norm(block, state, device):
    """(scale, bias) of block.bn3 for an input on ``device``, or None (stock path).  The fold is recomputed on every call (a few
    [C]-sized ops, no synchronisation): a training-mode BatchNorm2d forward updates running_mean / running_var in place without
    bumping their version counters, and writes through ``.data`` bypass them too, so no cached value could be trusted.  Only the
    probe, which checks that the module's forward IS ``x * scale + bias``, is keyed on the tensors' addresses and versions."""
    norm = block.bn3
    kind = _norm_kind(norm)
    if kind is None:
        return None
    tensors = _norm_tensors(norm, kind)
    if not all(isinstance(t, torch.Tensor) and t.device == device and t.dtype == torch.float32 for t in tensors):
        return None
    scale, bias = _fold(norm, kind)
    key = (type(norm), kind, getattr(norm, "eps", None)) + tuple((t.data_ptr(), t._version) for t in tensors)
    if key != state.key:
        state.key, state.ok = key, _probe_ok(norm, kind, scale, bias)
        if not state.ok and not state.warned:
            warnings.warn(f"fuse_backbone_tail: {type(norm).__name__}.forward differs from the folded x * scale + bias; "
                          "the block keeps its stock forward", RuntimeWarning, stacklevel=3)
            state.warned = True
    return (scale, bias) if state.ok else None


def _stock_forward(block, state, x):
    if state.had_forward:
        return state.old_forward(x)
    return type(block).forward(block, x)


def _fused_forward(block, state, x):
    """Bottleneck.forward with the tail after conv3 (resnet.py:106-113) as one seam-format kernel."""
    fold = None
    if isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and block.conv3.out_channels % 8 == 0:
        fold = _folded_norm(block, state, x.device)
    if fold is None:
        return _stock_forward(block, state, x)
    identity = x
    out = block.relu(block.bn1(block.conv1(x)))
    out = block.relu(block.bn2(block.conv2(out)))
    c = block.conv3(out)
    if block.downsample is not None:
        identity = block.downsample(x)
    if c.dtype != torch.float32 or identity.dtype != torch.float32 or identity.shape != c.shape:
        # (autocast and friends) finish with the stock tail's own operations
        out = block.bn3(c)
        out += identity
        return block.relu(out)
    scale, bias = fold
    return ops.seam_tail(c, identity, scale, bias)


def _installed(block):
    fwd = block.__dict__.get("forward")
    return fwd if isinstance(fwd, _FusedForward) else None


def fuse_backbone_tail(feature_extractor: nn.Module) -> nn.Module:
    """Make the last Bottleneck of ``feature_extractor`` emit bf16 channels_last features (see the module docstring).  Returns
    ``feature_extractor``; a second call is a no-op.  Raises ValueError when no Bottleneck-shaped module is found.
    The hook lives in the block's instance __dict__: ``nn.DataParallel`` replicas (which copy that dict) would run it on the
    original block, so use one process per GPU (DistributedDataParallel), as the reference's trainers do."""
    block = _last_bottleneck(feature_extractor)
    if block is None:
        raise ValueError("fuse_backbone_tail: no module with conv1/bn1/conv2/bn2/conv3/bn3/relu/downsample (a Bottleneck) found")
    if _installed(block) is None:
        had = "forward" in block.__dict__
        block.__dict__["forward"] = _FusedForward(block, had, block.__dict__.get("forward"))
    return feature_extractor


def unfuse_backbone_tail(feature_extractor: nn.Module) -> nn.Module:
    """Restore the forward the last Bottleneck had before ``fuse_backbone_tail``."""
    block = _last_bottleneck(feature_extractor)
    state = None if block is None else _installed(block)
    if state is None:
        return feature_extractor
    if state.had_forward:
        block.__dict__["forward"] = state.old_forward
    else:
        del block.__dict__["forward"]
    return feature_extractor


def is_fused(feature_extractor: nn.Module) -> bool:
    block = _last_bottleneck(feature_extractor)
    return block is not None and _installed(block) is not None


def wrap_feature_extractor_factory(stock):
    """``build_feature_extractor`` with the same signature whose result goes through ``fuse_backbone_tail`` (install(seam=True))."""
    if getattr(stock, "_b200seg_seam", False):
        return stock

    @functools.wraps(stock)
    def build_feature_extractor(*args, **kwargs):
        fe = stock(*args, **kwargs)
        if isinstance(fe, nn.Module) and _last_bottleneck(fe) is not None:       # (a VGG backbone stays as built)
            fuse_backbone_tail(fe)
        return fe

    build_feature_extractor._b200seg_seam = True
    return build_feature_extractor
