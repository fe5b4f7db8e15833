"""Autograd-aware functional ops over the C ABI (the layer the nn.Modules are built from)."""
from __future__ import annotations

from typing import Optional, Sequence

import torch

from . import _lib


# --------------------------------------------------------------------------------------------
# K1  fused multi-dilation ASPP head
# --------------------------------------------------------------------------------------------
# The same feature tensor is consumed by several modules per iteration (FADA: classifier(tgt_fea) and model_D(tgt_fea),
# classifier(src_fea) and model_D(src_fea.detach()), aspp_fada.py:91-123), and each would convert it to the bf16 pixel-major
# GEMM operand again (an HBM pass of 12 B per element).  An OPT-IN LRU (``set_feature_pack_cache(n)``, default off) keeps the
# last conversions.  An entry holds a reference to the source storage (through a detached alias), so its address cannot be
# handed to another tensor while the entry lives, and it is keyed on the version counter, so any in-place update through
# torch invalidates it -- but NOT writes through ``.data``, raw pointers or CUDA-graph replays into a static buffer, which is
# why it is off unless the caller (who knows how the features are produced) turns it on; it also pins the fp32 sources.
_PACK_CACHE_SLOTS = 0
_pack_cache = []            # [(key, source alias, Xp)]


def set_feature_pack_cache(slots: int):
    """Number of converted feature tensors kept (0 disables the cache and drops the entries)."""
    global _PACK_CACHE_SLOTS
    _PACK_CACHE_SLOTS = max(0, int(slots))
    del _pack_cache[_PACK_CACHE_SLOTS:]


def clear_feature_pack_cache():
    del _pack_cache[:]


def _pixel_major_bf16(x: torch.Tensor) -> torch.Tensor:
    """[N,Cin,h,w] -> bf16 [N*h*w, Cin].  bf16 channels_last input is taken zero-copy."""
    if not x.is_cuda:
        raise _lib.B200SegError("ASPP head: expected CUDA features (b200seg has no CPU fallback)")
    N, Cin, h, w = x.shape
    if x.dtype == torch.bfloat16:
        xl = x.permute(0, 2, 3, 1)
        if not xl.is_contiguous():
            xl = xl.contiguous()
        return xl.reshape(N * h * w, Cin)
    if x.dtype != torch.float32:
        x = x.float()
    x = x.contiguous()
    if _PACK_CACHE_SLOTS <= 0:
        return _lib.aspp_pack_features(x)
    key = (x.data_ptr(), x._version, tuple(x.shape), x.device.index, _lib._stream(x.device))
    for i, (k, _, Xp) in enumerate(_pack_cache):
        if k == key:
            _pack_cache.insert(0, _pack_cache.pop(i))
            return Xp
    Xp = _lib.aspp_pack_features(x)
    _pack_cache.insert(0, (key, x.detach(), Xp))
    del _pack_cache[_PACK_CACHE_SLOTS:]
    return Xp


def _fused_convert_ok(x: torch.Tensor, C: int, R: int) -> bool:
    """fp32 NCHW features can go straight into the forward GEMM (conversion in its producer warps, no pack pass) -- unless the
    caller turned the cross-module conversion cache on, in which case the packed copy is wanted for the other consumers."""
    return _PACK_CACHE_SLOTS <= 0 and x.is_cuda and x.dtype == torch.float32 and _lib.aspp_forward_f32_supported(x.contiguous(), C, R)


class _AsppHeadFn(torch.autograd.Function):
    """out[N,C,h,w] = sum_r conv3x3(x; W_r, b_r, dilation=padding=rates[r])  (classifier.py:26-29)."""

    @staticmethod
    def forward(ctx, x, rates, packed, need_w, *params):
        R = len(rates)
        weights, biases = params[:R], params[R:]
        N, Cin, h, w = x.shape
        C = weights[0].shape[0]
        if packed is None:
            packed = _lib.aspp_pack_weights([p.detach() for p in weights], [None if b is None else b.detach() for b in biases])
        Wp, WpT, bias_sum = packed
        ctx.rates, ctx.shape, ctx.x_dtype = tuple(rates), (N, Cin, h, w, C), x.dtype
        if not need_w and _fused_convert_ok(x, C, R):
            # eval / frozen head: straight from the fp32 NCHW features, no pack pass and nothing of x kept for backward
            logits, _ = _lib.aspp_forward_f32(x.detach().contiguous(), Wp, bias_sum, rates, C)
            ctx.save_for_backward(None, WpT)
            return logits
        Xp = _pixel_major_bf16(x.detach())
        logits = _lib.aspp_forward(Xp, Wp, bias_sum, rates, N, h, w, C)
        ctx.save_for_backward(Xp, WpT)
        return logits

    @staticmethod
    def backward(ctx, grad_logits):
        Xp, WpT = ctx.saved_tensors
        N, Cin, h, w, C = ctx.shape
        R = len(ctx.rates)
        need = ctx.needs_input_grad          # x, rates, packed, need_w, R weights, R biases
        need_x = need[0]
        need_w = any(need[4:4 + R])
        need_b = any(need[4 + R:4 + 2 * R])
        gx, gws, gbs = _lib.aspp_backward(grad_logits.float(), Xp, WpT, ctx.rates, N, h, w, C, need_x, need_w, need_b)
        if gx is not None and ctx.x_dtype != torch.float32:
            gx = gx.to(ctx.x_dtype)
        out_w = [gws[r] if (gws is not None and need[4 + r]) else None for r in range(R)]
        out_b = [gbs[r] if (gbs is not None and need[4 + R + r]) else None for r in range(R)]
        return (gx, None, None, None, *out_w, *out_b)


def aspp_head(x: torch.Tensor, weights: Sequence[torch.Tensor], biases: Sequence[Optional[torch.Tensor]],
              rates: Sequence[int], packed=None) -> torch.Tensor:
    need_w = torch.is_grad_enabled() and any(p.requires_grad for p in weights)
    return _AsppHeadFn.apply(x, tuple(int(r) for r in rates), packed, need_w, *weights, *biases)


class _AsppHeadLossFn(torch.autograd.Function):
    """Fused train slice: head forward -> upsample + CE forward, and in backward CE/upsample backward -> head dgrad /
    wgrad with the low-res gradient handed over as packed bf16 (no fp32 NCHW gradient, no transposes).  ONE foreign call per
    direction (b200seg_head_loss_forward / _backward): weight pack, feature pack, GEMMs, gathers and reductions are enqueued from
    C, with one workspace allocation that lives from forward to backward."""

    @staticmethod
    def forward(ctx, x, labels, ignore_index, temperature, rates, grad_bucket, *params):
        R = len(rates)
        ctx.grad_bucket = grad_bucket
        weights, biases = params[:R], params[R:]
        N, Cin, h, w = x.shape
        C = weights[0].shape[0]
        xd = x.detach()
        if not xd.is_cuda:
            raise _lib.B200SegError("ASPP head: expected CUDA features (b200seg has no CPU fallback)")
        if xd.dtype == torch.bfloat16 or _PACK_CACHE_SLOTS > 0:
            xk, x_kind = _pixel_major_bf16(xd), 1           # bf16 channels_last input is taken zero-copy
        else:
            xk, x_kind = (xd if xd.dtype == torch.float32 else xd.float()).contiguous(), 0
        need_grad = any(ctx.needs_input_grad)
        inv_t = 1.0 / float(temperature)
        # (only the parameters' addresses cross the boundary: no detached views needed)
        loss, logits, ws = _lib.head_loss_forward(xk, x_kind, (N, Cin, h, w), weights, biases, rates, labels.contiguous(),
                                                  ignore_index, inv_t, need_grad)
        ctx.meta = (rates, (N, Cin, h, w), C, tuple(labels.shape[-2:]), inv_t, x.dtype, need_grad, x_kind)
        ctx.save_for_backward(ws, xk if x_kind == 1 else None)
        ctx.mark_non_differentiable(logits)
        ctx.set_materialize_grads(False)       # no zero tensor for the (non-differentiable) logits output in backward
        return loss, logits

    @staticmethod
    def backward(ctx, grad_loss, _grad_logits_unused):
        ws, x_bf16 = ctx.saved_tensors
        rates, shape, C, size, inv_t, x_dtype, need_grad, x_kind = ctx.meta
        if not need_grad:
            raise _lib.B200SegError("forward_loss: forward ran without gradient tracking")
        R = len(rates)
        need = ctx.needs_input_grad          # x, labels, ignore_index, temperature, rates, grad_bucket, R weights, R biases
        need_w = any(need[6:6 + R])
        need_b = any(need[6 + R:6 + 2 * R])
        if grad_loss is None:
            return (None,) * (6 + 2 * R)
        grad_loss = grad_loss.detach()
        if grad_loss.dtype != torch.float32:
            grad_loss = grad_loss.float()
        # bf16 features (the channels_last seam format): the dgrad GEMM writes the bf16 NHWC gradient itself
        seam = x_dtype == torch.bfloat16 and shape[1] % 8 == 0
        bucket = ctx.grad_bucket
        if bucket is not None and need_w and need_b:
            # data-parallel path: the weight / bias gradients are written straight into the flat bucket (the parameters'
            # .grad alias it), and the bucket's all-reduce starts on its own stream as soon as they are complete --
            # underneath the data-gradient GEMM.  Autograd gets no parameter gradients from this node.
            gx, _, _ = _lib.head_loss_backward(ws, x_bf16, x_kind, shape, C, rates, size, inv_t, grad_loss, need[0], True, True,
                                               nhwc_bf16=seam, out_w=bucket.weight_buffers(), out_b=bucket.bias_buffers(),
                                               weights_ready_event=bucket.ready_event)
            bucket.begin_allreduce_()
            if gx is not None and gx.dtype != x_dtype:
                gx = gx.to(x_dtype)
            return (gx,) + (None,) * (5 + 2 * R)
        gx, gws, gbs = _lib.head_loss_backward(ws, x_bf16, x_kind, shape, C, rates, size, inv_t, grad_loss, need[0], need_w, need_b,
                                               nhwc_bf16=seam)
        if gx is not None and gx.dtype != x_dtype:
            gx = gx.to(x_dtype)
        out_w = [gws[r] if (gws is not None and need[6 + r]) else None for r in range(R)]
        out_b = [gbs[r] if (gbs is not None and need[6 + R + r]) else None for r in range(R)]
        return (gx, None, None, None, None, None, *out_w, *out_b)


def aspp_head_loss(x, labels, weights, biases, rates, ignore_index=255, temperature=1.0, packed=None, grad_bucket=None):
    """(loss, low-res logits [detached]) == CrossEntropyLoss(ignore_index)(interpolate(head(x), labels.shape[-2:]) / T, labels).
    ``grad_bucket`` (distributed.HeadGradBucket): write the parameter gradients into the bucket and overlap its all-reduce
    with the data-gradient GEMM instead of returning them through autograd.  ``packed`` is accepted for compatibility and
    ignored: the weights are packed inside the one-call entry on every step (a ~6 us kernel), never cached."""
    labels = _lib.as_label_tensor(labels)            # int64 or uint8 as they are; anything else widened to int64
    return _AsppHeadLossFn.apply(x, labels, int(ignore_index), float(temperature), tuple(int(r) for r in rates), grad_bucket,
                                 *weights, *biases)


# --------------------------------------------------------------------------------------------
# K6  PixelDiscriminator conv stack (three 3x3 layers as tcgen05 implicit GEMMs, bf16 NHWC activations)
# --------------------------------------------------------------------------------------------
def pack_discriminator_weights(w1, w2, wc1, wc2, bc1, bc2):
    """((Wf1, Wb1), (Wf2, Wb2), (Wf3, Wb3), bias3) -- cls1 | cls2 are packed as ONE layer with 2C output channels (the
    torch.cat of discriminator.py:47 costs nothing)."""
    C = wc1.shape[0]
    (l1, l2, l3), b3 = _lib.conv3x3_pack_weights_stack(
        [[w1.detach()], [w2.detach()], [wc1.detach(), wc2.detach()]],
        bias_parts=[None if bc1 is None else bc1.detach(), None if bc2 is None else bc2.detach()], bias_lens=[C, C])     # ONE launch
    return l1, l2, l3, b3


class _PixelDiscriminatorFn(torch.autograd.Function):
    """cat(cls1(mid), cls2(mid)) with mid = LReLU(conv(LReLU(conv(x))))  (discriminator.py:34-47), fp32 NCHW [N,2C,h,w].
    ONE foreign call per direction (b200seg_disc_forward / _backward, graph-replayed in a steady-state loop)."""

    @staticmethod
    def forward(ctx, x, slope, packed, w1, b1, w2, b2, wc1, bc1, wc2, bc2):
        N, Cin, h, w = x.shape
        xd = x.detach()
        if not xd.is_cuda:
            raise _lib.B200SegError("PixelDiscriminator: expected CUDA features (b200seg has no CPU fallback)")
        if xd.dtype == torch.bfloat16 or _PACK_CACHE_SLOTS > 0:
            xk, x_kind = _pixel_major_bf16(xd).view(N, h, w, Cin), 1          # bf16 channels_last input is taken zero-copy
        else:
            xk, x_kind = (xd if xd.dtype == torch.float32 else xd.float()).contiguous(), 0
        out, Xp, A1, A2, packed = _lib.disc_forward(xk, x_kind, (N, Cin, h, w), (w1, w2, wc1, wc2), (b1, b2, bc1, bc2), slope, packed)
        (_, Wb1), (_, Wb2), (_, Wb3), _ = packed
        ctx.meta = (float(slope), x.dtype, int(wc1.shape[0]))
        ctx.save_for_backward(Xp, A1, A2, Wb1, Wb2, Wb3)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        Xp, A1, A2, Wb1, Wb2, Wb3 = ctx.saved_tensors
        slope, x_dtype, C = ctx.meta
        need = ctx.needs_input_grad          # x, slope, packed, w1, b1, w2, b2, wc1, bc1, wc2, bc2
        go = grad_out.detach()
        if go.dtype != torch.float32:
            go = go.float()
        gx, gw1, gb1, gw2, gb2, gwc1, gbc1, gwc2, gbc2 = _lib.disc_backward(
            go.contiguous(), Xp, A1, A2, Wb1, Wb2, Wb3, C, slope, (need[0],) + tuple(need[3:11]), x_bf16=(x_dtype == torch.bfloat16))
        if gx is not None and gx.dtype != x_dtype:
            gx = gx.to(x_dtype)
        return gx, None, None, gw1, gb1, gw2, gb2, gwc1, gbc1, gwc2, gbc2


def pixel_discriminator_logits(x, w1, b1, w2, b2, wc1, bc1, wc2, bc2, slope: float = 0.2, packed=None) -> torch.Tensor:
    return _PixelDiscriminatorFn.apply(x, float(slope), packed, w1, b1, w2, b2, wc1, bc1, wc2, bc2)


# --------------------------------------------------------------------------------------------
# seam-format producer: the last Bottleneck's bn3 + residual + relu, emitted as bf16 channels_last
# --------------------------------------------------------------------------------------------
class _SeamTailFn(torch.autograd.Function):
    """bf16 channels_last relu((c * scale + bias) + identity)  (resnet.py:106-113 with a folded FrozenBatchNorm2d, layers.py:17-23).
    Saves only y (and the [C] scale): when the head consumes y it keeps the same storage as its GEMM operand, so the stock tail's
    fp32 relu output is not kept at all."""

    @staticmethod
    def forward(ctx, c, identity, scale, bias):
        y = _lib.seam_tail_forward(c.detach().contiguous(), identity.detach().contiguous(), scale.detach().contiguous(),
                                   bias.detach().contiguous())
        ctx.save_for_backward(y, scale.detach())
        return y

    @staticmethod
    def backward(ctx, dy):
        y, scale = ctx.saved_tensors
        need_c, need_id = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        dy = dy.detach()
        # the head's seam-format dgrad already writes bf16 channels_last; a sum of two consumers' gradients or the NCHW bf16
        # gradient of the plain head call is converted once
        if dy.dtype != torch.bfloat16 or not dy.is_contiguous(memory_format=torch.channels_last):
            dy = dy.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        dc, di = _lib.seam_tail_backward(dy, y, scale.contiguous(), need_c, need_id)
        return dc, di, None, None


def seam_tail(c: torch.Tensor, identity: torch.Tensor, scale: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """bf16 channels_last ``relu((c * scale + bias) + identity)`` from fp32 NCHW ``c`` / ``identity`` [N, C, h, w] (C % 8 == 0)
    and the folded norm's fp32 ``scale`` / ``bias`` [C] (constants: no gradient).  Bit-identical to the stock fp32 sequence
    followed by ``.to(torch.bfloat16)``; the gradient to ``c`` / ``identity`` is the stock one computed from the bf16 ``dy``."""
    return _SeamTailFn.apply(c, identity, scale, bias)


# --------------------------------------------------------------------------------------------
# materialising align-corners bilinear upsample (API-compat path)
# --------------------------------------------------------------------------------------------
class _UpsampleFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, size):
        ctx.in_hw = tuple(x.shape[-2:])
        return _lib.upsample_bilinear_forward(x.detach().float().contiguous(), size)

    @staticmethod
    def backward(ctx, grad_out):
        return _lib.upsample_bilinear_backward(grad_out.float(), ctx.in_hw), None


def upsample_bilinear_align_corners(x: torch.Tensor, size) -> torch.Tensor:
    """F.interpolate(x, size, mode='bilinear', align_corners=True), bit-exact forward on CUDA."""
    return _UpsampleFn.apply(x, (int(size[0]), int(size[1])))


# --------------------------------------------------------------------------------------------
# K2  upsample + cross-entropy (ignore_index), fused
# --------------------------------------------------------------------------------------------
class _UpsampleCEFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits_lr, labels, ignore_index, temperature):
        need_grad = bool(ctx.needs_input_grad[0])
        inv_t = 1.0 / float(temperature)
        out2, ws = _lib.upsample_ce_forward(logits_lr.detach().float().contiguous(), labels.contiguous(), ignore_index, inv_t,
                                            need_grad)
        ctx.meta = (tuple(logits_lr.shape), tuple(labels.shape[-2:]), inv_t, need_grad)
        ctx.save_for_backward(out2, ws)
        return out2[0].clone()

    @staticmethod
    def backward(ctx, grad_out):
        out2, ws = ctx.saved_tensors
        shape_lr, size, inv_t, need_grad = ctx.meta
        if not need_grad:
            raise _lib.B200SegError("upsample_cross_entropy: forward ran without gradient tracking")
        g = _lib.upsample_ce_backward(ws, out2, shape_lr, size, inv_t, grad_out.detach().float())
        return g, None, None, None


def upsample_cross_entropy(logits_lr: torch.Tensor, labels: torch.Tensor, ignore_index: int = 255,
                           temperature: float = 1.0) -> torch.Tensor:
    """CrossEntropyLoss(ignore_index)(interpolate(logits_lr, labels.shape[-2:]) / temperature, labels) without
    materialising the full-resolution logits (aspp_trainer.py:88-92, aspp_fada.py:91-96)."""
    labels = _lib.as_label_tensor(labels)
    return _UpsampleCEFn.apply(logits_lr, labels, int(ignore_index), float(temperature))


# --------------------------------------------------------------------------------------------
# K3  soft-label cross-entropy
# --------------------------------------------------------------------------------------------
class _SoftCEFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, soft, weights):
        pred_c = pred.detach().float().contiguous()
        soft_c = soft.detach().float().contiguous()
        w_c = None if weights is None else weights.detach().float().contiguous()
        loss, stats = _lib.soft_ce_forward(pred_c, soft_c, w_c, want_stats=bool(ctx.needs_input_grad[0]))
        ctx.save_for_backward(pred_c, soft_c, w_c, stats)
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        pred_c, soft_c, w_c, stats = ctx.saved_tensors
        return _lib.soft_ce_backward(pred_c, soft_c, w_c, grad_out.detach().float(), stats), None, None


def soft_label_cross_entropy(pred: torch.Tensor, soft_label: torch.Tensor,
                             pixel_weights: Optional[torch.Tensor] = None) -> torch.Tensor:
    """core/utils/utility.py:172-177 (differentiable w.r.t. pred only, as every reference caller uses it).  Lazy operands
    (lazy.py: the discriminator's un-materialised output against a soft label built from un-materialised head logits,
    aspp_fada.py:110-124) take the fused K6 + K5 path; anything else is materialised and streamed through K3."""
    from . import lazy
    if lazy.is_lazy(pred) or lazy.is_lazy(soft_label):
        fused = lazy.soft_label_loss(pred, soft_label, pixel_weights)
        if fused is not NotImplemented:
            return fused
        pred, soft_label = lazy.materialize(pred), lazy.materialize(soft_label)
    return _SoftCEFn.apply(pred, soft_label, pixel_weights)


# --------------------------------------------------------------------------------------------
# K5  fused FADA discriminator loss tail (upsample + soft-label build + soft-label CE on low-res tensors)
# --------------------------------------------------------------------------------------------
class _FadaSoftCEFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, d_logits, seg_logits, size, slot, temperature, clamp):
        need_grad = bool(ctx.needs_input_grad[0])
        out2, ws = _lib.fada_softce_forward(d_logits.detach().float().contiguous(), seg_logits.detach().float().contiguous(), size,
                                            slot, 1.0 / float(temperature), clamp, need_grad)
        ctx.meta = (tuple(d_logits.shape), tuple(size), need_grad)
        ctx.save_for_backward(out2, ws)
        return out2[0].clone()

    @staticmethod
    def backward(ctx, grad_out):
        out2, ws = ctx.saved_tensors
        shape_d, size, need_grad = ctx.meta
        if not need_grad:
            raise _lib.B200SegError("fada_soft_label_loss: forward ran without gradient tracking")
        return _lib.fada_softce_backward(ws, out2, shape_d, size, grad_out.detach().float()), None, None, None, None, None


def fada_soft_label_loss(d_logits_lr: torch.Tensor, seg_logits_lr: torch.Tensor, size, slot: int, temperature: float = 1.8,
                         clamp: float = 0.9) -> torch.Tensor:
    """soft_label_cross_entropy(interpolate(d_logits_lr, size), q) with q = min(softmax(interpolate(seg_logits_lr, size) / T), clamp)
    placed in the source slot (0: cat(q, 0)) or the target slot (1: cat(0, q)) -- the three discriminator losses of
    aspp_fada.py:110-125 -- computed on the low-resolution tensors only.  seg_logits_lr is treated as a constant
    (the reference detaches the soft labels); the gradient flows to d_logits_lr."""
    C = seg_logits_lr.shape[1]
    if not _lib.fada_softce_supported(C):        # more than 32 classes (K2 / K4 do not take those either): materialised operands + K3
        up_d = upsample_bilinear_align_corners(d_logits_lr, size)
        with torch.no_grad():
            soft = torch.softmax(upsample_bilinear_align_corners(seg_logits_lr, size) / temperature, dim=1)
            soft = torch.clamp(soft, max=clamp)
            zeros = torch.zeros_like(soft)
            q = torch.cat((soft, zeros) if slot == 0 else (zeros, soft), dim=1)
        return soft_label_cross_entropy(up_d, q)
    return _FadaSoftCEFn.apply(d_logits_lr, seg_logits_lr, (int(size[0]), int(size[1])), int(slot), float(temperature), float(clamp))
