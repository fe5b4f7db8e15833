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
norm's current tensors on every call.  Anything else -- another norm, a failed probe, and by default a training-mode
BatchNorm2d / SyncBatchNorm -- runs the block's stock forward.

Batch statistics (opt-in: ``fuse_backbone_tail(fe, train_bn=True)`` / ``install(seam=True, seam_train_bn=True)``): a ``bn3`` that
is exactly ``nn.BatchNorm2d`` or ``nn.SyncBatchNorm`` in training mode with running statistics runs ops.seam_tail_bn: the batch
mean / variance, the running-statistics update and ``relu(((c - mean) * invstd * weight + bias) + identity)`` as bf16
channels_last, with the gradient to c, identity and the norm's weight / bias.  A SyncBatchNorm whose group (``process_group`` or
the world) has more than one rank exchanges its statistics over that group, which must be NCCL; otherwise it is per-rank, as
in SyncBatchNorm.forward.  The statistics match PyTorch's to fp32 rounding, not bit for bit.  The flag also lets an eval-mode
SyncBatchNorm with constant affine parameters take the fold.  Subclasses, ``track_running_stats=False``, another backend, a
single value per channel, autocast and CPU input keep the stock forward.

conv3 fused into the tail (opt-in: ``fuse_backbone_tail(fe, conv3=True)`` / ``install(seam=True, seam_conv3=True)``): when the fold
applies (a 'frozen' or 'bn' bn3 as above) and ``conv3`` is exactly ``nn.Conv2d`` -- 1x1, stride 1, padding 0, groups 1, no bias,
an fp32 weight on the input's device, Cin % 8 == 0 and Cout % 8 == 0 -- and conv2's output is fp32, the block runs
ops.seam_conv3_tail: conv3 as a tcgen05 GEMM whose epilogue applies the fold, the residual and the relu and writes the bf16
channels_last features, so conv3's fp32 output is neither written nor read back.  Numerics: conv2's output and conv3's weight are
each rounded to bf16 once and accumulated in fp32 (the head's standing choice), the tail is applied to the fp32 accumulator in the
fold's order and rounded once to bf16; the features are therefore NOT bit-identical to the stock block's, unlike the fold path.
The backward computes conv3's data gradient from bf16(scale * weight) and its weight gradient from bf16(out2), with fp32
accumulation.  Every other case (a training-mode 'batch' bn3 included: see below) takes the path above with a stock conv3.

conv3 under batch statistics (opt-in: ``fuse_backbone_tail(fe, train_bn=True, conv3_batch=True)`` / ``install(seam=True,
seam_train_bn=True, seam_conv3_batch=True)``): when bn3 takes the batch-statistics path above and conv3 is eligible as for
``conv3=True``, conv2's output and the identity are fp32 of the expected shape and there is more than one value per channel, the
block runs ops.seam_conv3_tail_bn: conv3 as a tcgen05 GEMM that writes its fp32 NCHW output c once and computes the per-rank
statistics from its accumulator (no pass reads c back for them), then the batch tail above, unchanged.  Numerics: conv2's output
and conv3's weight are each rounded to bf16 once with fp32 accumulation; the statistics are those of the stored c; in the
backward, the gradient into c is rounded once to bf16 before conv3's data and weight gradient GEMMs.  ``conv3=True`` keeps its
meaning (the fold only); everything else keeps the batch path with a stock conv3.
"""
from __future__ import annotations

import functools
import warnings

import torch
import torch.distributed as dist
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
    tensors) under which the fold last passed or failed its probe, and ``train_bn`` / ``conv3`` / ``conv3_batch``
    (fuse_backbone_tail's flags)."""
    train_bn = False                    # (objects pickled before a flag existed load with the default)
    conv3 = False
    conv3_batch = False

    def __init__(self, block, had_forward, old_forward, train_bn=False, conv3=False, conv3_batch=False):
        self.block, self.had_forward, self.old_forward = block, had_forward, old_forward
        self.key, self.ok, self.warned = None, False, False
        self.train_bn = bool(train_bn)
        self.conv3 = bool(conv3)
        self.conv3_batch = bool(conv3_batch)

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


def _norm_kind(norm, train_bn=False):
    """'frozen', 'bn' (eval-mode BatchNorm2d with constant affine parameters in this call) or None (stays stock).  With
    ``train_bn`` also 'batch' (exactly nn.BatchNorm2d / nn.SyncBatchNorm in training mode with running statistics), and an
    eval-mode SyncBatchNorm is taken like an eval-mode BatchNorm2d."""
    if train_bn and type(norm) in (nn.BatchNorm2d, nn.SyncBatchNorm) and norm.training:
        if norm.track_running_stats and norm.running_mean is not None and norm.running_var is not None:
            return "batch"
        return None
    if isinstance(norm, nn.BatchNorm2d) or (train_bn and isinstance(norm, nn.SyncBatchNorm)):
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
    kind = _norm_kind(norm, state.train_bn)
    if kind not in ("frozen", "bn"):
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


def _batch_group(norm, device):
    """For a 'batch' norm: (group,) with the process group to exchange statistics over (None: this rank's batch only), or None
    when the norm stays stock (tensors elsewhere or of another dtype, a group that is not NCCL)."""
    tensors = [t for t in (norm.weight, norm.bias, norm.running_mean, norm.running_var) if t is not None]
    if not all(t.device == device and t.dtype == torch.float32 for t in tensors):
        return None
    nbt = norm.num_batches_tracked
    if nbt is not None and (nbt.device != device or nbt.dtype != torch.int64):
        return None
    if isinstance(norm, nn.SyncBatchNorm) and dist.is_available() and dist.is_initialized():
        group = norm.process_group or dist.group.WORLD
        if dist.get_world_size(group) > 1:
            return (group,) if dist.get_backend(group) == "nccl" else None
    return (None,)


def _conv3_fusable(conv, x):
    """conv3 can run inside the fused GEMM: exactly nn.Conv2d, 1x1, stride 1, no padding, one group, no bias, an fp32 weight on x's
    device, input and output channels multiples of 8."""
    return (type(conv) is nn.Conv2d and conv.kernel_size == (1, 1) and conv.stride == (1, 1) and conv.padding in ((0, 0), "valid")
            and conv.groups == 1 and conv.bias is None and conv.weight.dtype == torch.float32 and conv.weight.device == x.device
            and conv.in_channels % 8 == 0 and conv.out_channels % 8 == 0)


def _stock_forward(block, state, x):
    if state.had_forward:
        return state.old_forward(x)
    return type(block).forward(block, x)


def _fused_forward(block, state, x):
    """Bottleneck.forward with the tail after conv3 (resnet.py:106-113) as one seam-format kernel."""
    fold = batch = None
    if isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and block.conv3.out_channels % 8 == 0:
        if _norm_kind(block.bn3, state.train_bn) == "batch":
            batch = _batch_group(block.bn3, x.device)
        else:
            fold = _folded_norm(block, state, x.device)
    if fold is None and batch is None:
        return _stock_forward(block, state, x)
    identity = x
    out = block.relu(block.bn1(block.conv1(x)))
    out = block.relu(block.bn2(block.conv2(out)))
    if fold is not None and state.conv3 and out.dtype == torch.float32 and _conv3_fusable(block.conv3, x):
        if block.downsample is not None:
            identity = block.downsample(x)
        if identity.dtype == torch.float32 and tuple(identity.shape) == (out.shape[0], block.conv3.out_channels) + tuple(out.shape[2:]):
            return ops.seam_conv3_tail(out, identity, block.conv3.weight, fold[0], fold[1])
        c = block.conv3(out)
    elif batch is not None and state.conv3_batch and out.dtype == torch.float32 and _conv3_fusable(block.conv3, x):
        if block.downsample is not None:
            identity = block.downsample(x)
        shape = (out.shape[0], block.conv3.out_channels) + tuple(out.shape[2:])
        single = batch[0] is None and out.shape[0] * out.shape[2] * out.shape[3] <= 1
        if identity.dtype == torch.float32 and tuple(identity.shape) == shape and not single:
            norm = block.bn3
            return ops.seam_conv3_tail_bn(out, identity, block.conv3.weight, norm.weight, norm.bias, norm.running_mean,
                                          norm.running_var, norm.num_batches_tracked, norm.momentum, norm.eps, batch[0])
        c = block.conv3(out)
    else:
        c = block.conv3(out)
        if block.downsample is not None:
            identity = block.downsample(x)
    single = batch is not None and batch[0] is None and c.numel() <= c.shape[1]
    if c.dtype != torch.float32 or identity.dtype != torch.float32 or identity.shape != c.shape or single:
        # (autocast and friends; one value per channel, which the stock norm rejects) finish with the stock tail's own operations
        out = block.bn3(c)
        out += identity
        return block.relu(out)
    if batch is not None:
        norm = block.bn3
        return ops.seam_tail_bn(c, identity, norm.weight, norm.bias, norm.running_mean, norm.running_var, norm.num_batches_tracked,
                                norm.momentum, norm.eps, batch[0])
    scale, bias = fold
    return ops.seam_tail(c, identity, scale, bias)


def _installed(block):
    fwd = block.__dict__.get("forward")
    return fwd if isinstance(fwd, _FusedForward) else None


def fuse_backbone_tail(feature_extractor: nn.Module, train_bn: bool = False, conv3: bool = False,
                       conv3_batch: bool = False) -> nn.Module:
    """Make the last Bottleneck of ``feature_extractor`` emit bf16 channels_last features (see the module docstring).  Returns
    ``feature_extractor``; a second call only sets ``train_bn`` (a training-mode BatchNorm2d / SyncBatchNorm bn3 takes the
    batch-statistics kernels), ``conv3`` (an eligible conv3 runs inside the fused GEMM, with bf16 operands: see the module
    docstring for what that changes numerically) and ``conv3_batch`` (with ``train_bn``: an eligible conv3 of a batch-statistics
    bn3 runs as a tcgen05 GEMM that writes its output and statistics, also with bf16 operands).  Raises ValueError when no Bottleneck-shaped module is found.
    The hook lives in the block's instance __dict__: ``nn.DataParallel`` replicas (which copy that dict) would run it on the
    original block, so use one process per GPU (DistributedDataParallel), as the reference's trainers do."""
    block = _last_bottleneck(feature_extractor)
    if block is None:
        raise ValueError("fuse_backbone_tail: no module with conv1/bn1/conv2/bn2/conv3/bn3/relu/downsample (a Bottleneck) found")
    state = _installed(block)
    if state is None:
        had = "forward" in block.__dict__
        block.__dict__["forward"] = _FusedForward(block, had, block.__dict__.get("forward"), train_bn, conv3, conv3_batch)
    else:
        state.train_bn = bool(train_bn)
        state.conv3 = bool(conv3)
        state.conv3_batch = bool(conv3_batch)
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


def wrap_feature_extractor_factory(stock, train_bn: bool = False, conv3: bool = False, conv3_batch: bool = False):
    """``build_feature_extractor`` with the same signature whose result goes through ``fuse_backbone_tail(fe, train_bn, conv3,
    conv3_batch)`` (install(seam=True, seam_train_bn=..., seam_conv3=..., seam_conv3_batch=...)).  Wrapping a wrapper returns it
    with its flags set to the new values."""
    if getattr(stock, "_b200seg_seam", False):
        stock._b200seg_seam_train_bn = bool(train_bn)
        stock._b200seg_seam_conv3 = bool(conv3)
        stock._b200seg_seam_conv3_batch = bool(conv3_batch)
        return stock

    @functools.wraps(stock)
    def build_feature_extractor(*args, **kwargs):
        fe = stock(*args, **kwargs)
        if isinstance(fe, nn.Module) and _last_bottleneck(fe) is not None:       # (a VGG backbone stays as built)
            fuse_backbone_tail(fe, train_bn=build_feature_extractor._b200seg_seam_train_bn,
                               conv3=build_feature_extractor._b200seg_seam_conv3,
                               conv3_batch=build_feature_extractor._b200seg_seam_conv3_batch)
        return fe

    build_feature_extractor._b200seg_seam = True
    build_feature_extractor._b200seg_seam_train_bn = bool(train_bn)
    build_feature_extractor._b200seg_seam_conv3 = bool(conv3)
    build_feature_extractor._b200seg_seam_conv3_batch = bool(conv3_batch)
    return build_feature_extractor
