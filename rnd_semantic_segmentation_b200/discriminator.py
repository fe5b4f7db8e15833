"""PixelDiscriminator -- drop-in for core/models/discriminator.py:31-50.

Parameter owners and state_dict keys (``D.0``, ``D.2``, ``cls1``, ``cls2``) are identical to the
reference (real ``nn.Conv2d`` children, created in the same order with the default init).  The
arithmetic is NOT cuDNN: the three 3x3 layers run as tcgen05 implicit GEMMs on bf16 NHWC activations
with bias / LeakyReLU / LeakyReLU-backward fused into the epilogues (csrc/conv_sm100.cu, SURVEY.md
section 8f rank 1), cls1 | cls2 as ONE layer with 2C outputs written as fp32 NCHW; then the tail --
align-corners upsample, or the fused soft-label loss (``forward_soft_loss``).  ``D.tf32 = True`` runs the
same GEMMs with TF32 operands and fp32 activations / gradients (INTEGRATION.md "TF32 discriminator").
"""
from __future__ import annotations

import os

import torch
from torch import nn

from . import ops


class PixelDiscriminator(nn.Module):
    # tf32 = True: the conv stack runs with TF32 tensor-core operands and stores its activations and inter-layer gradients as fp32
    # (the numeric class of cuDNN under torch.backends.cudnn.allow_tf32) instead of bf16.  A plain attribute, not in state_dict(),
    # so checkpoints of both precisions are interchangeable; the class default covers modules pickled before the flag existed.
    tf32 = False

    def __init__(self, input_nc, ndf=512, num_classes=1):
        super().__init__()
        self.D = nn.Sequential(
            nn.Conv2d(input_nc, ndf, kernel_size=3, stride=1, padding=1),
            nn.LeakyReLU(negative_slope=0.2, inplace=True),
            nn.Conv2d(ndf, ndf // 2, kernel_size=3, stride=1, padding=1),
            nn.LeakyReLU(negative_slope=0.2, inplace=True))
        self.cls1 = nn.Conv2d(ndf // 2, num_classes, kernel_size=3, stride=1, padding=1)
        self.cls2 = nn.Conv2d(ndf // 2, num_classes, kernel_size=3, stride=1, padding=1)

        self._packed = None
        self._packed_key = None
        self.lazy = None        # None = automatic (lazy.lazy_enabled): lazy unless a multi-rank process group is initialised
        self.tf32 = False

    def out_channels_lowres(self):
        return int(self.cls1.out_channels + self.cls2.out_channels)

    def _params(self):
        return [self.D[0].weight, self.D[0].bias, self.D[2].weight, self.D[2].bias,
                self.cls1.weight, self.cls1.bias, self.cls2.weight, self.cls2.bias]

    def invalidate_packed(self):
        """Drop the cached weight pack (see ASPP_Classifier_V2.invalidate_packed)."""
        self._packed = None
        self._packed_key = None

    def _packed_weights(self):
        """Packed weights of the three layers (bf16, or TF32 values in fp32 with ``tf32``): re-packed on every call in training mode
        (one launch; version counters miss ``.data`` / raw-pointer / graph-replay writes), cached on (precision, data_ptr, _version)
        in eval mode only."""
        params = self._params()
        tf32 = bool(self.tf32)
        key = (tf32,) + tuple((p.data_ptr(), p._version) for p in params)
        if self.training or self._packed is None or key != self._packed_key:
            w1, _, w2, _, wc1, bc1, wc2, bc2 = params
            self._packed = ops.pack_discriminator_weights(w1, w2, wc1, wc2, bc1, bc2, tf32=tf32)
            self._packed_key = key
        return self._packed

    def logits(self, x):
        """Low-resolution logits [N,2C,h,w] = cat(cls1(D(x)), cls2(D(x)))  (discriminator.py:45-47)."""
        # training mode: the weights are packed INSIDE the one-call forward on every call (version counters miss ``.data`` /
        # raw-pointer / graph-replay writes); eval mode reuses the pack cached on (data_ptr, _version)
        return ops.pixel_discriminator_logits(x, *self._params(), slope=self.D[1].negative_slope,
                                              packed=None if self.training else self._packed_weights(), tf32=bool(self.tf32))

    def forward(self, x, size=None):
        from . import lazy as _lazy
        if size is not None and x.is_cuda and _lazy.lazy_enabled(self.lazy):                  # discriminator.py:48-49, evaluated by its consumer
            from .lazy import LazyLogits, _LogitsSource
            return LazyLogits(_LogitsSource(self, x, size))
        out = self.logits(x)
        if size is not None:                                              # discriminator.py:48-49
            out = ops.upsample_bilinear_align_corners(out, size)
        return out

    # ---- fused extension ------------------------------------------------------------------
    def forward_soft_loss(self, x, seg_logits_lr, size, slot, temperature: float = 1.8, clamp: float = 0.9):
        """soft_label_cross_entropy(self(x, size), cat-slot(min(softmax(interpolate(seg_logits_lr, size) / T), clamp)))
        -- aspp_fada.py:110-111 (slot 0), :119-120 (slot 0), :123-124 (slot 1) -- without any full-resolution tensor."""
        return ops.fada_soft_label_loss(self.logits(x), seg_logits_lr, size, slot, temperature, clamp)
