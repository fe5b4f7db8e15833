"""ctypes binding of libb200seg.so (C ABI declared in include/b200seg.h).

PyTorch is used for device memory and streams only: every wrapper below takes
CUDA tensors, checks dtype / contiguity / device, and hands raw device pointers
plus the current CUDA stream to the C entry point.  There is no CPU fallback:
a missing library or a CPU tensor raises.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional, Sequence

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
# B200SEG_LIB selects another build of the same library (kernel A/B experiments under profiles/)
LIB_PATH = os.environ.get("B200SEG_LIB") or os.path.join(_PKG, "libb200seg.so")
_lib = None

c_int, c_i64, c_f32, c_vp = ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p

# name -> (restype, argtypes); must list every symbol include/b200seg.h declares
SIGNATURES = {
    "b200seg_abi_version": (c_int, []),
    "b200seg_last_error": (ctypes.c_char_p, []),
    "b200seg_device_sms": (c_int, []),
    "b200seg_upsample_argmax_confusion": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_int, c_int, c_vp, c_i64,
                                                  c_vp, c_int, c_vp]),
    "b200seg_upsample_argmax_confusion_ex": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_i64,
                                                     c_vp, c_int, c_int, c_vp]),
    "b200seg_upsample_argmax_confusion_frames": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp,
                                                         c_i64, c_vp, c_int, c_vp]),
    "b200seg_confusion_from_pred": (c_int, [c_vp, c_vp, c_i64, c_int, c_int, c_int, c_vp, c_vp]),
    "b200seg_confusion_from_pred_ex": (c_int, [c_vp, c_int, c_vp, c_int, c_i64, c_int, c_int, c_int, c_vp, c_vp]),
    "b200seg_upsample_ce_forward_ex": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_int, c_int, c_int, c_f32, c_int, c_vp,
                                               c_i64, c_vp, c_vp]),
    "b200seg_tta_argmax_confusion_ex": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_int, c_vp, c_int,
                                                c_int, c_vp, c_vp, c_int, c_vp, c_vp]),
    "b200seg_upsample_ce_workspace_bytes": (c_i64, [c_int] * 6),
    "b200seg_upsample_ce_forward": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_int, c_int, c_f32, c_int, c_vp,
                                            c_i64, c_vp, c_vp]),
    "b200seg_upsample_ce_set_variant": (None, [c_int]),
    "b200seg_p2p_allreduce_mean": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_i64, c_int, c_int, c_vp]),
    "b200seg_upsample_ce_backward": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_f32, c_vp, c_vp, c_vp, c_vp]),
    "b200seg_upsample_ce_backward_packed": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "b200seg_upsample_bilinear_forward": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp]),
    "b200seg_upsample_bilinear_backward": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp]),
    "b200seg_soft_ce_workspace_bytes": (c_i64, []),
    "b200seg_soft_ce_forward": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_i64, c_vp, c_vp]),
    "b200seg_soft_ce_backward": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp]),
    "b200seg_soft_ce_stats_bytes": (c_i64, [c_int, c_int, c_int]),
    "b200seg_soft_ce_forward_stats": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "b200seg_soft_ce_backward_stats": (c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp]),
    "b200seg_fada_softce_workspace_bytes": (c_i64, [c_int] * 6),
    "b200seg_fada_softce_forward": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_f32, c_f32, c_int, c_int, c_vp, c_i64,
                                            c_vp, c_vp]),
    "b200seg_fada_softce_backward": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp]),
    "b200seg_aspp_packed_rows": (c_int, [c_int, c_int]),
    "b200seg_aspp_pack_weights": (c_int, [c_vp, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp]),
    "b200seg_aspp_pack_features": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp]),
    "b200seg_aspp_forward_scratch_bytes": (c_i64, [c_int] * 5),
    "b200seg_aspp_forward": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp]),
    "b200seg_aspp_forward_f32_supported": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_int]),
    "b200seg_aspp_forward_f32": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp]),
    "b200seg_gemm_set_fwd_convert": (None, [c_int]),
    "b200seg_gemm_set_dgrad_mode": (None, [c_int]),
    "b200seg_gemm_set_fwd_mode": (None, [c_int]),
    "b200seg_gemm_fwd_convert_selftest": (c_int, [c_int] * 5 + [ctypes.POINTER(ctypes.c_double)] * 3),
    "b200seg_aspp_backward_scratch_bytes": (c_i64, [c_int] * 7),
    "b200seg_aspp_backward": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_i64, c_int,
                                      c_vp, c_vp, c_vp, c_vp]),
    "b200seg_aspp_backward_packed": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_i64, c_int,
                                             c_vp, c_vp, c_vp]),
    "b200seg_aspp_backward_packed_nhwc": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_i64,
                                                  c_int, c_vp, c_vp, c_vp]),
    "b200seg_aspp_backward_packed_ex": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_i64,
                                                c_int, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "b200seg_head_loss_workspace_bytes": (c_i64, [c_int] * 9),
    "b200seg_head_loss_scratch_bytes": (c_i64, [c_int] * 6),
    "b200seg_head_loss_forward": (c_int, [c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_int, c_int,
                                          c_int, c_int, c_f32, c_int, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "b200seg_head_loss_backward": (c_int, [c_vp, c_i64, c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                           c_f32, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "b200seg_aspp_default_wgrad_splits": (c_int, [c_i64, c_int, c_int, c_int]),
    "b200seg_disc_backward_scratch_bytes": (c_i64, [c_int] * 7),
    "b200seg_disc_forward": (c_int, [c_vp, c_int] + [c_int] * 7 + [c_vp] * 8 + [c_f32, c_int] + [c_vp] * 11 + [c_vp]),
    "b200seg_disc_backward": (c_int, [c_vp] * 7 + [c_int] * 7 + [c_f32] + [c_vp] * 4 + [c_i64] + [c_vp] * 9 + [c_vp]),
    "b200seg_set_step_graphs": (None, [c_int]),
    "b200seg_step_graph_stats": (None, [c_vp, c_vp]),
    "b200seg_conv3x3_pack_weights": (c_int, [c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_int, c_vp]),
    "b200seg_conv3x3_pack_weights_stack": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp]),
    "b200seg_conv3x3_forward": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_i64, c_vp, c_int, c_int, c_vp, c_int, c_f32, c_vp, c_i64,
                                        c_vp, c_vp]),
    "b200seg_conv3x3_dgrad": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_i64, c_vp, c_int, c_int, c_vp, c_f32, c_vp, c_i64, c_vp,
                                      c_vp]),
    "b200seg_conv3x3_dgrad_colsum_scratch_bytes": (c_i64, [c_int, c_int, c_int, c_i64]),
    "b200seg_conv3x3_dgrad_colsum": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_i64, c_vp, c_int, c_int, c_vp, c_f32, c_vp, c_i64,
                                             c_vp, c_i64, c_vp, c_vp]),
    "b200seg_conv3x3_wgrad_scratch_bytes": (c_i64, [c_int] * 6),
    "b200seg_conv3x3_wgrad": (c_int, [c_vp, c_int, c_i64, c_vp, c_int, c_i64, c_int, c_int, c_int, c_int, c_int, c_vp, c_i64, c_vp,
                                      c_vp, c_int, c_vp]),
    "b200seg_nchw_to_nhwc_bf16": (c_int, [c_vp, c_int, c_int, c_int, c_vp, c_int, c_vp]),
    "b200seg_seam_tail_forward": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_vp]),
    "b200seg_seam_tail_backward": (c_int, [c_vp, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp]),
    "b200seg_nhwc_colsum_scratch_bytes": (c_i64, [c_int]),
    "b200seg_nhwc_bf16_colsum": (c_int, [c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_vp]),
    "b200seg_gemm_set_overlap_sms": (None, [c_int]),
    "b200seg_launch_count": (ctypes.c_longlong, []),
    "b200seg_profile_enable": (None, [c_int]),
    "b200seg_profile_read": (c_int, [c_int, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(c_int)]),
    "b200seg_gemm_selftest": (c_int, [c_int] * 8 + [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]),
    "b200seg_gemm_set_sharing": (None, [c_int]),
    "b200seg_conv_set_pair": (None, [c_int]),
    "b200seg_gemm_set_narrow_tiles": (None, [c_int]),
    "b200seg_tta_argmax_confusion": (c_int, [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_vp, c_int, c_int,
                                             c_vp, c_vp, c_vp, c_vp]),
    "b200seg_tta_set_row_walk": (None, [c_int]),
    "b200seg_sgd_step": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_f32, c_f32, c_f32, c_f32, c_int, c_int, c_f32, c_vp]),
    "b200seg_adam_step": (c_int, [c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_f32, c_f32, c_f32, c_f32, c_f32, c_i64, c_f32, c_vp]),
}


class B200SegError(RuntimeError):
    pass


def load(build_if_missing: bool = False) -> ctypes.CDLL:
    """Load the shared library (once).  Fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if build_if_missing:
            from ._build_ext import build
            build()
        else:
            raise B200SegError(
                f"{LIB_PATH} not found: build it with `python -m rnd_semantic_segmentation_b200._build_ext` "
                "(or __graft_entry__.build()).  There is no CPU / PyTorch fallback for this path.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    if lib.b200seg_abi_version() != 1:
        raise B200SegError("libb200seg.so ABI version mismatch")
    _lib = lib
    if os.environ.get("B200SEG_GEMM_SHARING"):        # A/B experiments (profiles/): operand-sharing mode of the head GEMMs
        lib.b200seg_gemm_set_sharing(int(os.environ["B200SEG_GEMM_SHARING"]))
    if os.environ.get("B200SEG_GEMM_NARROW"):
        lib.b200seg_gemm_set_narrow_tiles(int(os.environ["B200SEG_GEMM_NARROW"]))
    if os.environ.get("B200SEG_FWD_CONVERT"):
        lib.b200seg_gemm_set_fwd_convert(int(os.environ["B200SEG_FWD_CONVERT"]))
    if os.environ.get("B200SEG_CONV_PAIR"):
        lib.b200seg_conv_set_pair(int(os.environ["B200SEG_CONV_PAIR"]))
    return lib


def _check(rc: int):
    if rc != 0:
        raise B200SegError(load().b200seg_last_error().decode("utf-8", "replace"))


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream(device=None) -> int:
    """cudaStream_t of torch's current stream (on ``device``, default: the current device).  The raw getter costs a fraction
    of a microsecond; torch.cuda.current_stream() builds a Stream object and resolves the device index (~15 us) -- with a
    dozen launches per step that alone was 0.1 ms of host time per step."""
    if device is not None and not isinstance(device, int):
        device = device.index
    if device is None:
        device = torch.cuda.current_device()
    if _raw_stream is not None:
        return _raw_stream(device)
    return torch.cuda.current_stream(device).cuda_stream


class _on_device:
    """``with _on_device(dev)`` only when ``dev`` is not already current (the context manager costs ~10 us a call)."""
    __slots__ = ("ctx",)

    def __init__(self, device):
        idx = device.index if device.index is not None else torch.cuda.current_device()
        self.ctx = None if idx == torch.cuda.current_device() else torch.cuda.device(idx)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)
        return False


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor, got {type(t)}")
    if not t.is_cuda:
        raise B200SegError(f"{name}: expected a CUDA tensor (b200seg has no CPU fallback), got device {t.device}")
    if t.dtype != dtype:
        raise B200SegError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise B200SegError(f"{name}: expected a contiguous tensor")
    return t


def device_sms() -> int:
    return load().b200seg_device_sms()


LABEL_DTYPES = (torch.int64, torch.uint8)


def as_label_tensor(t: torch.Tensor) -> torch.Tensor:
    """Label / prediction maps are consumed as int64 (what the reference passes after ``.long()``, aspp_trainer.py:86,
    aspp_tester.py:58) or as uint8 (the tensor the dataloader holds, core/datasets/transform.py:31-33) without a conversion
    pass; any other integer dtype is widened to int64 first."""
    return t if t.dtype in LABEL_DTYPES else t.long()


def _need_label(t: torch.Tensor, name: str) -> int:
    """Checks a label / prediction map and returns its element width in bytes (8 or 1)."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor, got {type(t)}")
    if not t.is_cuda:
        raise B200SegError(f"{name}: expected a CUDA tensor (b200seg has no CPU fallback), got device {t.device}")
    if t.dtype not in LABEL_DTYPES:
        raise B200SegError(f"{name}: expected dtype torch.int64 or torch.uint8, got {t.dtype}")
    if not t.is_contiguous():
        raise B200SegError(f"{name}: expected a contiguous tensor")
    return 8 if t.dtype == torch.int64 else 1


def _pred_dtype(want_pred):
    """want_pred: False / True (int64, the reference's max(1)[1]) / torch.uint8 / torch.int64."""
    if want_pred is True:
        return torch.int64
    if want_pred in LABEL_DTYPES:
        return want_pred
    if not want_pred:
        return None
    raise B200SegError(f"want_pred: expected a bool, torch.int64 or torch.uint8, got {want_pred!r}")


# --------------------------------------------------------------------------------------------
# K4
# --------------------------------------------------------------------------------------------
def upsample_argmax_confusion(logits_lr: torch.Tensor, labels: Optional[torch.Tensor], size, num_classes: Optional[int] = None,
                              ignore_index: int = 255, cm: Optional[torch.Tensor] = None, per_frame: bool = False,
                              want_pred=False, fma_mode: int = 0):
    """Returns (cm, pred).  cm int64 [C,C] (or [N,C,C] if per_frame) accumulated in place when given.  ``labels``: int64 or
    uint8 [N,H,W]; ``want_pred``: True (int64) or torch.uint8 / torch.int64."""
    lib = load()
    _need(logits_lr, torch.float32, "logits")
    N, C, h, w = logits_lr.shape
    H, W = int(size[0]), int(size[1])
    if num_classes is not None and num_classes != C:
        raise B200SegError(f"logits have {C} channels but num_classes={num_classes}")
    lbytes = 8
    if labels is not None:
        lbytes = _need_label(labels, "labels")
        if labels.numel() != N * H * W:
            raise B200SegError(f"labels shape {tuple(labels.shape)} does not match N*H*W = {N}*{H}*{W}")
    stride = 0
    if labels is not None:
        if cm is None:
            cm = torch.zeros((N, C, C) if per_frame else (C, C), dtype=torch.int64, device=logits_lr.device)
        _need(cm, torch.int64, "cm")
        stride = C * C if cm.dim() == 3 else 0
    pdt = _pred_dtype(want_pred)
    pred = torch.empty((N, H, W), dtype=pdt, device=logits_lr.device) if pdt is not None else None
    with _on_device(logits_lr.device):
        _check(lib.b200seg_upsample_argmax_confusion_ex(logits_lr.data_ptr(), N, C, h, w, _ptr(labels), lbytes, H, W, ignore_index,
                                                        _ptr(cm) if labels is not None else None, stride, _ptr(pred),
                                                        1 if pdt == torch.uint8 else 8, fma_mode, _stream()))
    return cm, pred


def upsample_argmax_confusion_frames(logits: Sequence[torch.Tensor], labels: Optional[Sequence[torch.Tensor]], size,
                                     ignore_index: int = 255, cm: Optional[torch.Tensor] = None, per_frame: bool = False,
                                     want_pred=False):
    """K4 over several frames of the tester loop in ONE launch (16 frames per kernel launch): ``logits[f]`` fp32 [C,h,w] (or
    [1,C,h,w]) and ``labels[f]`` int64 / uint8 [H,W] are separate tensors (no concatenation pass).  Returns (cm, [pred_f] | None)
    with cm int64 [C,C] accumulated over the frames, or [F,C,C] with ``per_frame``."""
    lib = load()
    F_ = len(logits)
    if F_ == 0:
        raise B200SegError("upsample_argmax_confusion_frames: no frames")
    maps = []
    for f, t in enumerate(logits):
        _need(t, torch.float32, f"logits[{f}]")
        if t.dim() == 4 and t.shape[0] == 1:
            t = t[0]
        if t.dim() != 3 or (maps and t.shape != maps[0].shape) or t.device != logits[0].device:
            raise B200SegError(f"logits[{f}]: expected one [C,h,w] map per frame, all of one shape and device")
        maps.append(t)
    C, h, w = (int(v) for v in maps[0].shape)
    H, W = int(size[0]), int(size[1])
    dev = maps[0].device
    lbytes = 8
    if labels is not None:
        if len(labels) != F_:
            raise B200SegError("upsample_argmax_confusion_frames: one label map per frame")
        lbytes = _need_label(labels[0], "labels[0]")
        for f, t in enumerate(labels):
            if _need_label(t, f"labels[{f}]") != lbytes or t.numel() != H * W or t.device != dev:
                raise B200SegError(f"labels[{f}]: expected {H}x{W} maps of one dtype on {dev}")
        if cm is None:
            cm = torch.zeros((F_, C, C) if per_frame else (C, C), dtype=torch.int64, device=dev)
        _need(cm, torch.int64, "cm")
    elif cm is not None:
        raise B200SegError("upsample_argmax_confusion_frames: a confusion matrix needs labels")
    stride = C * C if (cm is not None and cm.dim() == 3) else 0
    pdt = _pred_dtype(want_pred)
    preds = [torch.empty((H, W), dtype=pdt, device=dev) for _ in range(F_)] if pdt is not None else None
    with _on_device(dev):
        _check(lib.b200seg_upsample_argmax_confusion_frames(_ptr_array(maps), F_, C, h, w,
                                                            _ptr_array(list(labels)) if labels is not None else None, lbytes, H, W,
                                                            ignore_index, _ptr(cm), stride,
                                                            _ptr_array(preds) if preds is not None else None,
                                                            1 if pdt == torch.uint8 else 8, _stream()))
    return cm, preds


def tta_argmax_confusion(members: Sequence[torch.Tensor], flips: Sequence[bool], size, labels: Optional[torch.Tensor] = None,
                         divisors: Sequence[float] = (), ignore_index: int = 255, cm: Optional[torch.Tensor] = None,
                         want_pred=False, want_probs: bool = False, div_exact: bool = False):
    """K7: fused test-time augmentation for ONE frame.  ``members``: fp32 [C,h_m,w_m] (or [1,C,h_m,w_m]) low-res logit maps,
    ``flips[m]``: member m was computed on the mirrored image.  Returns (cm | None, pred int64 [H,W] | None, probs fp32 [C,H,W] | None)
    with probs = (sum_m unflip(softmax(upsample(member_m)))) / divisors[0] [/ divisors[1]] and pred its first argmax."""
    lib = load()
    if len(members) == 0 or len(members) != len(flips):
        raise B200SegError("tta_argmax_confusion: members and flips must be non-empty and of equal length")
    maps = []
    for m, t in enumerate(members):
        _need(t, torch.float32, f"members[{m}]")
        if t.dim() == 4 and t.shape[0] == 1:
            t = t[0]
        if t.dim() != 3:
            raise B200SegError(f"members[{m}]: expected [C,h,w] or [1,C,h,w], got {tuple(t.shape)}")
        if maps and t.shape[0] != maps[0].shape[0]:
            raise B200SegError("tta_argmax_confusion: members disagree on the number of classes")
        if t.device != members[0].device:
            raise B200SegError("tta_argmax_confusion: members must live on one device")
        maps.append(t)
    C = int(maps[0].shape[0])
    H, W = int(size[0]), int(size[1])
    dev = maps[0].device
    lbytes = 8
    if labels is not None:
        lbytes = _need_label(labels, "labels")
        if labels.numel() != H * W:
            raise B200SegError(f"labels shape {tuple(labels.shape)} does not match H*W = {H}*{W}")
        if cm is None:
            cm = torch.zeros((C, C), dtype=torch.int64, device=dev)
        _need(cm, torch.int64, "cm")
    elif cm is not None:
        raise B200SegError("tta_argmax_confusion: a confusion matrix needs labels")
    if len(divisors) > 2:
        raise B200SegError("tta_argmax_confusion: at most two divisors")
    pdt = _pred_dtype(want_pred)
    pred = torch.empty((H, W), dtype=pdt, device=dev) if pdt is not None else None
    probs = torch.empty((C, H, W), dtype=torch.float32, device=dev) if want_probs else None
    n = len(maps)
    hs = (c_int * n)(*[int(t.shape[1]) for t in maps])
    ws = (c_int * n)(*[int(t.shape[2]) for t in maps])
    fl = (c_int * n)(*[1 if f else 0 for f in flips])
    dv = (c_f32 * max(1, len(divisors)))(*[float(d) for d in divisors])
    with _on_device(dev):
        _check(lib.b200seg_tta_argmax_confusion_ex(_ptr_array(maps), hs, ws, fl, n, C, _ptr(labels), lbytes, H, W, int(ignore_index),
                                                   dv, len(divisors), 1 if div_exact else 0, _ptr(cm), _ptr(pred),
                                                   1 if pdt == torch.uint8 else 8, _ptr(probs), _stream()))
    return cm, pred, probs


def tta_set_row_walk(on, fast: bool = True):
    """K7 A/B: row-walking kernel for <= 4 members (default) vs the per-pixel kernel; ``fast=False`` disables the labels-only
    fast path of the row-walking kernel (approximate ordering + exact fallback on near ties)."""
    load().b200seg_tta_set_row_walk((1 if on else 0) | (0 if fast else 2))


def _optim_tables(params, grads, *states):
    n = len(params)
    for i, (p, g) in enumerate(zip(params, grads)):
        _need(p, torch.float32, f"params[{i}]")
        _need(g, torch.float32, f"grads[{i}]")
        if g.numel() != p.numel() or g.device != p.device:
            raise B200SegError(f"optimizer step: gradient {i} does not match its parameter")
    for st in states:
        if st is None:
            continue
        if len(st) != n:
            raise B200SegError("optimizer step: state list length != number of parameters")
        for i, (p, b) in enumerate(zip(params, st)):
            _need(b, torch.float32, f"state[{i}]")
            if b.numel() != p.numel() or b.device != p.device:
                raise B200SegError(f"optimizer step: state tensor {i} does not match its parameter")
    numels = (c_i64 * n)(*[int(p.numel()) for p in params])
    return n, numels


def sgd_step(params: Sequence[torch.Tensor], grads: Sequence[torch.Tensor], momentum_bufs: Optional[Sequence[torch.Tensor]], lr: float,
             momentum: float = 0.0, dampening: float = 0.0, weight_decay: float = 0.0, nesterov: bool = False,
             first_step: bool = False, grad_scale: float = 1.0):
    """K8: torch.optim.SGD's update of a whole parameter group in one launch (in place on params / momentum_bufs)."""
    lib = load()
    if not params:
        return
    n, numels = _optim_tables(params, grads, momentum_bufs if momentum != 0 else None)
    with _on_device(params[0].device):
        _check(lib.b200seg_sgd_step(n, _ptr_array(params), _ptr_array(grads), _ptr_array(momentum_bufs) if momentum != 0 else None,
                                    numels, float(lr), float(momentum), float(dampening), float(weight_decay), 1 if nesterov else 0,
                                    1 if first_step else 0, float(grad_scale), _stream()))


def adam_step(params: Sequence[torch.Tensor], grads: Sequence[torch.Tensor], exp_avg: Sequence[torch.Tensor],
              exp_avg_sq: Sequence[torch.Tensor], step: int, lr: float, beta1: float = 0.9, beta2: float = 0.999, eps: float = 1e-8,
              weight_decay: float = 0.0, grad_scale: float = 1.0):
    """K8: torch.optim.Adam's update of a whole parameter group in one launch; ``step`` counts this update (>= 1)."""
    lib = load()
    if not params:
        return
    n, numels = _optim_tables(params, grads, exp_avg, exp_avg_sq)
    with _on_device(params[0].device):
        _check(lib.b200seg_adam_step(n, _ptr_array(params), _ptr_array(grads), _ptr_array(exp_avg), _ptr_array(exp_avg_sq), numels,
                                     float(lr), float(beta1), float(beta2), float(eps), float(weight_decay), int(step),
                                     float(grad_scale), _stream()))


def confusion_from_pred(pd: torch.Tensor, gt: torch.Tensor, num_classes: int, ignore_index: int = 255,
                        mutate_pd: bool = False, cm: Optional[torch.Tensor] = None) -> torch.Tensor:
    lib = load()
    pb = _need_label(pd, "pd")
    gb = _need_label(gt, "gt")
    if pd.numel() != gt.numel():
        raise B200SegError("pd and gt must have the same number of elements")
    if cm is None:
        cm = torch.zeros(num_classes, num_classes, dtype=torch.int64, device=pd.device)
    _need(cm, torch.int64, "cm")
    with _on_device(pd.device):
        _check(lib.b200seg_confusion_from_pred_ex(pd.data_ptr(), pb, gt.data_ptr(), gb, pd.numel(), num_classes, ignore_index,
                                                  1 if mutate_pd else 0, cm.data_ptr(), _stream()))
    return cm


# --------------------------------------------------------------------------------------------
# K2 + materialising upsample
# --------------------------------------------------------------------------------------------
def upsample_ce_forward(logits_lr, labels, ignore_index=255, inv_temperature=1.0, need_grad=True):
    """Returns (loss_and_count float32[2], workspace) -- workspace feeds upsample_ce_backward."""
    lib = load()
    _need(logits_lr, torch.float32, "logits")
    lbytes = _need_label(labels, "labels")
    N, C, h, w = logits_lr.shape
    H, W = labels.shape[-2:]
    if labels.numel() != N * H * W:
        raise B200SegError(f"labels shape {tuple(labels.shape)} does not match batch {N}")
    nbytes = lib.b200seg_upsample_ce_workspace_bytes(N, C, h, w, H, W)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=logits_lr.device)
    out2 = torch.empty(2, dtype=torch.float32, device=logits_lr.device)
    with _on_device(logits_lr.device):
        _check(lib.b200seg_upsample_ce_forward_ex(logits_lr.data_ptr(), N, C, h, w, labels.data_ptr(), lbytes, H, W, ignore_index,
                                                  float(inv_temperature), 1 if need_grad else 0, ws.data_ptr(), nbytes,
                                                  out2.data_ptr(), _stream()))
    return out2, ws


def p2p_allreduce_mean(peer_ptrs: Sequence[int], multicast_ptr: int, signal_pad_ptrs: Sequence[int], rank: int, world: int, numel: int,
                       blocks: int = 8, pad_slot0: int = 0, device=None):
    """Enqueue the peer-memory mean all-reduce kernel on the current stream of ``device`` (every rank must)."""
    lib = load()
    n = len(peer_ptrs)
    bufs = (c_vp * n)(*[int(v) for v in peer_ptrs])
    pads = (c_vp * n)(*[int(v) for v in signal_pad_ptrs])
    _check(lib.b200seg_p2p_allreduce_mean(bufs, int(multicast_ptr) if multicast_ptr else None, pads, int(rank), int(world), int(numel),
                                          int(blocks), int(pad_slot0), _stream(device)))


def upsample_ce_set_variant(v: int):
    """K2 A/B: 1 (default) = warp-tile kernel where eligible and measured faster (19 classes), 2 = wherever eligible (also 2
    classes), 0 = always the CTA-tile kernel."""
    load().b200seg_upsample_ce_set_variant(int(v))


def upsample_ce_backward(ws, out2, shape_lr, size, inv_temperature=1.0, grad_out: Optional[torch.Tensor] = None):
    lib = load()
    N, C, h, w = shape_lr
    H, W = size
    if grad_out is not None:
        grad_out = _need(grad_out.reshape(1).contiguous(), torch.float32, "grad_out")
    grad = torch.empty((N, C, h, w), dtype=torch.float32, device=ws.device)
    with _on_device(ws.device):
        _check(lib.b200seg_upsample_ce_backward(ws.data_ptr(), N, C, h, w, H, W, float(inv_temperature), out2.data_ptr(),
                                                _ptr(grad_out), grad.data_ptr(), _stream()))
    return grad


def upsample_ce_backward_packed(ws, out2, shape_lr, size, inv_temperature=1.0, grad_out: Optional[torch.Tensor] = None,
                                want_bias: bool = True):
    """Returns (gOt: bf16 low-res gradient as class planes [N][C][h*w] in a [N*h*w, 32] buffer, bias_grad fp32 [C] | None)."""
    lib = load()
    N, C, h, w = shape_lr
    H, W = size
    if grad_out is not None:
        grad_out = _need(grad_out.reshape(1).contiguous(), torch.float32, "grad_out")
    gOt = torch.empty((N * h * w, 32), dtype=torch.bfloat16, device=ws.device)
    bias = torch.empty(C, dtype=torch.float32, device=ws.device) if want_bias else None
    with _on_device(ws.device):
        _check(lib.b200seg_upsample_ce_backward_packed(ws.data_ptr(), N, C, h, w, H, W, float(inv_temperature), out2.data_ptr(),
                                                       _ptr(grad_out), gOt.data_ptr(), _ptr(bias), _stream()))
    return gOt, bias


def upsample_bilinear_forward(x: torch.Tensor, size, fma_mode: int = 0) -> torch.Tensor:
    lib = load()
    _need(x, torch.float32, "input")
    N, C, h, w = x.shape
    H, W = int(size[0]), int(size[1])
    out = torch.empty((N, C, H, W), dtype=torch.float32, device=x.device)
    with _on_device(x.device):
        _check(lib.b200seg_upsample_bilinear_forward(x.data_ptr(), out.data_ptr(), N * C, h, w, H, W, fma_mode, _stream()))
    return out


def upsample_bilinear_backward(grad_out: torch.Tensor, in_hw) -> torch.Tensor:
    lib = load()
    grad_out = _need(grad_out.contiguous(), torch.float32, "grad_output")
    N, C, H, W = grad_out.shape
    h, w = in_hw
    gin = torch.empty((N, C, h, w), dtype=torch.float32, device=grad_out.device)
    with _on_device(grad_out.device):
        _check(lib.b200seg_upsample_bilinear_backward(grad_out.data_ptr(), gin.data_ptr(), N * C, h, w, H, W, _stream()))
    return gin


# --------------------------------------------------------------------------------------------
# K3
# --------------------------------------------------------------------------------------------
def soft_ce_forward(pred, soft, weights=None, want_stats: bool = False):
    """loss (0-d); with ``want_stats`` also the per-pixel {lse, sum q} planes for soft_ce_backward (None when the shapes do
    not allow the vectorised path)."""
    lib = load()
    _need(pred, torch.float32, "pred")
    _need(soft, torch.float32, "soft_label")
    if pred.shape != soft.shape or pred.dim() != 4:
        raise B200SegError(f"pred {tuple(pred.shape)} and soft_label {tuple(soft.shape)} must be equal 4-d shapes")
    N, K, H, W = pred.shape
    if weights is not None:
        _need(weights, torch.float32, "pixel_weights")
        if weights.numel() != N * H * W:
            raise B200SegError("pixel_weights must have N*H*W elements")
    nbytes = lib.b200seg_soft_ce_workspace_bytes()
    ws = torch.empty(nbytes, dtype=torch.uint8, device=pred.device)
    out = torch.empty(1, dtype=torch.float32, device=pred.device)
    stats = None
    if want_stats and (H * W) % 4 == 0 and all(t is None or t.data_ptr() % 16 == 0 for t in (pred, soft, weights)):
        stats = torch.empty(lib.b200seg_soft_ce_stats_bytes(N, H, W) // 4, dtype=torch.float32, device=pred.device)
    with _on_device(pred.device):
        if stats is not None:
            _check(lib.b200seg_soft_ce_forward_stats(pred.data_ptr(), soft.data_ptr(), _ptr(weights), N, K, H, W, ws.data_ptr(),
                                                     nbytes, stats.data_ptr(), out.data_ptr(), _stream()))
        else:
            _check(lib.b200seg_soft_ce_forward(pred.data_ptr(), soft.data_ptr(), _ptr(weights), N, K, H, W, ws.data_ptr(), nbytes,
                                               out.data_ptr(), _stream()))
    return (out.reshape(()), stats) if want_stats else out.reshape(())


def soft_ce_backward(pred, soft, weights, grad_out, stats=None) -> torch.Tensor:
    lib = load()
    N, K, H, W = pred.shape
    grad_out = _need(grad_out.reshape(1).contiguous(), torch.float32, "grad_out")
    grad = torch.empty_like(pred)
    if stats is not None:
        with _on_device(pred.device):
            _check(lib.b200seg_soft_ce_backward_stats(pred.data_ptr(), soft.data_ptr(), _ptr(weights), stats.data_ptr(),
                                                      grad_out.data_ptr(), N, K, H, W, grad.data_ptr(), _stream()))
        return grad
    with _on_device(pred.device):
        _check(lib.b200seg_soft_ce_backward(pred.data_ptr(), soft.data_ptr(), _ptr(weights), grad_out.data_ptr(), N, K, H, W,
                                            grad.data_ptr(), _stream()))
    return grad


# --------------------------------------------------------------------------------------------
# K5  fused FADA discriminator loss tail
# --------------------------------------------------------------------------------------------
def fada_softce_supported(num_classes: int) -> bool:
    """The fused K5 kernel takes any class count up to 32 (compile-time instantiations for 19 and 2, padded ones otherwise)."""
    return 1 <= num_classes <= 32


def fada_softce_forward(d_logits, seg_logits, size, slot: int, inv_temperature: float, clamp: float, need_grad: bool = True):
    lib = load()
    _need(d_logits, torch.float32, "d_logits")
    _need(seg_logits, torch.float32, "seg_logits")
    N, K, h, w = d_logits.shape
    C = seg_logits.shape[1]
    if K != 2 * C or tuple(seg_logits.shape) != (N, C, h, w):
        raise B200SegError(f"d_logits {tuple(d_logits.shape)} must be [N,2C,h,w] for seg_logits {tuple(seg_logits.shape)}")
    H, W = int(size[0]), int(size[1])
    nbytes = lib.b200seg_fada_softce_workspace_bytes(N, C, h, w, H, W)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=d_logits.device)
    out2 = torch.empty(2, dtype=torch.float32, device=d_logits.device)
    with _on_device(d_logits.device):
        _check(lib.b200seg_fada_softce_forward(d_logits.data_ptr(), seg_logits.data_ptr(), N, C, h, w, H, W, float(inv_temperature),
                                               float(clamp), int(slot), 1 if need_grad else 0, ws.data_ptr(), nbytes,
                                               out2.data_ptr(), _stream()))
    return out2, ws


def fada_softce_backward(ws, out2, shape_d, size, grad_out: Optional[torch.Tensor] = None):
    lib = load()
    N, K, h, w = shape_d
    H, W = size
    if grad_out is not None:
        grad_out = _need(grad_out.reshape(1).contiguous(), torch.float32, "grad_out")
    grad = torch.empty((N, K, h, w), dtype=torch.float32, device=ws.device)
    with _on_device(ws.device):
        _check(lib.b200seg_fada_softce_backward(ws.data_ptr(), N, K // 2, h, w, H, W, out2.data_ptr(), _ptr(grad_out),
                                                grad.data_ptr(), _stream()))
    return grad


# --------------------------------------------------------------------------------------------
# K1
# --------------------------------------------------------------------------------------------
def _ptr_array(tensors: Sequence[Optional[torch.Tensor]]):
    arr = (c_vp * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = None if t is None else t.data_ptr()
    return arr


def aspp_packed_rows(C: int, R: int) -> int:
    return load().b200seg_aspp_packed_rows(C, R)


def aspp_pack_weights(weights: Sequence[torch.Tensor], biases: Sequence[Optional[torch.Tensor]]):
    """R x [C,Cin,3,3] fp32 (+ R x [C]) -> (Wp bf16 [NJ,Cin], WpT bf16 [Cin,NJ], bias_sum fp32 [C])."""
    lib = load()
    R = len(weights)
    C, Cin = weights[0].shape[:2]
    for wt in weights:
        _need(wt, torch.float32, "conv weight")
        if tuple(wt.shape) != (C, Cin, 3, 3):
            raise B200SegError(f"conv weight shape {tuple(wt.shape)} != {(C, Cin, 3, 3)}")
    for b in biases:
        if b is not None:
            _need(b, torch.float32, "conv bias")
    dev = weights[0].device
    NJ = lib.b200seg_aspp_packed_rows(C, R)
    Wp = torch.empty((NJ, Cin), dtype=torch.bfloat16, device=dev)
    WpT = torch.empty((Cin, NJ), dtype=torch.bfloat16, device=dev)
    bias_sum = torch.empty(C, dtype=torch.float32, device=dev)
    with _on_device(dev):
        _check(lib.b200seg_aspp_pack_weights(_ptr_array(weights), _ptr_array(biases), R, C, Cin, Wp.data_ptr(), WpT.data_ptr(),
                                             bias_sum.data_ptr(), _stream()))
    return Wp, WpT, bias_sum


def aspp_pack_features(x: torch.Tensor) -> torch.Tensor:
    """fp32 NCHW [N,Cin,h,w] -> bf16 pixel-major [N*h*w, Cin]."""
    lib = load()
    _need(x, torch.float32, "features")
    N, Cin, h, w = x.shape
    Xp = torch.empty((N * h * w, Cin), dtype=torch.bfloat16, device=x.device)
    with _on_device(x.device):
        _check(lib.b200seg_aspp_pack_features(x.data_ptr(), N, Cin, h, w, Xp.data_ptr(), _stream()))
    return Xp


_scratch_cache = {}


def _scratch(key, nbytes: int, device) -> torch.Tensor:
    """Grow-only scratch per (purpose, device, STREAM): reuse is ordered by the stream it is used on (contents never outlive
    one op), and ops issued concurrently on different streams never share a buffer."""
    dev_index = device.index if device.index is not None else torch.cuda.current_device()
    k = (key, dev_index, _stream(dev_index))
    t = _scratch_cache.get(k)
    if t is None or t.numel() < nbytes:
        t = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
        _scratch_cache[k] = t
    return t


def aspp_forward(Xp: torch.Tensor, Wp: torch.Tensor, bias_sum: torch.Tensor, rates: Sequence[int], N: int, h: int, w: int,
                 C: int) -> torch.Tensor:
    lib = load()
    _need(Xp, torch.bfloat16, "Xp")
    _need(Wp, torch.bfloat16, "Wp")
    _need(bias_sum, torch.float32, "bias_sum")
    Cin = Xp.shape[1]
    R = len(rates)
    if Xp.shape[0] != N * h * w:
        raise B200SegError("Xp rows != N*h*w")
    nbytes = lib.b200seg_aspp_forward_scratch_bytes(N, C, h, w, R)
    scratch = _scratch("aspp_fwd", nbytes, Xp.device)
    logits = torch.empty((N, C, h, w), dtype=torch.float32, device=Xp.device)
    rates_arr = (c_int * R)(*[int(r) for r in rates])
    with _on_device(Xp.device):
        _check(lib.b200seg_aspp_forward(Xp.data_ptr(), Wp.data_ptr(), bias_sum.data_ptr(), rates_arr, R, N, Cin, C, h, w,
                                        scratch.data_ptr(), logits.data_ptr(), _stream()))
    return logits


def aspp_forward_f32_supported(x: torch.Tensor, C: int, R: int) -> bool:
    """True when the head's forward can take these fp32 NCHW features through the GEMM with in-kernel conversion."""
    if x.dtype != torch.float32 or not x.is_cuda or not x.is_contiguous() or x.dim() != 4:
        return False
    N, Cin, h, w = x.shape
    return bool(load().b200seg_aspp_forward_f32_supported(x.data_ptr(), Cin, C, h, w, R))


def aspp_forward_f32(x: torch.Tensor, Wp: torch.Tensor, bias_sum: torch.Tensor, rates: Sequence[int], C: int, want_xn: bool = False):
    """Head forward straight from fp32 NCHW features (no pack pass).  Returns (logits fp32 [N,C,h,w], xn bf16 [N,Cin,h,w] | None)."""
    lib = load()
    _need(x, torch.float32, "features")
    _need(Wp, torch.bfloat16, "Wp")
    _need(bias_sum, torch.float32, "bias_sum")
    N, Cin, h, w = x.shape
    R = len(rates)
    nbytes = lib.b200seg_aspp_forward_scratch_bytes(N, C, h, w, R)
    scratch = _scratch("aspp_fwd", nbytes, x.device)
    logits = torch.empty((N, C, h, w), dtype=torch.float32, device=x.device)
    xn = torch.empty((N, Cin, h, w), dtype=torch.bfloat16, device=x.device) if want_xn else None
    rates_arr = (c_int * R)(*[int(r) for r in rates])
    with _on_device(x.device):
        _check(lib.b200seg_aspp_forward_f32(x.data_ptr(), Wp.data_ptr(), bias_sum.data_ptr(), rates_arr, R, N, Cin, C, h, w,
                                            scratch.data_ptr(), logits.data_ptr(), _ptr(xn), _stream()))
    return logits, xn


def gemm_fwd_convert_selftest(M, n_img, hw, K, write_xn=True):
    lib = load()
    err, ref, xe = ctypes.c_double(0), ctypes.c_double(0), ctypes.c_double(0)
    _check(lib.b200seg_gemm_fwd_convert_selftest(M, n_img, hw, K, int(write_xn), ctypes.byref(err), ctypes.byref(ref), ctypes.byref(xe)))
    return err.value, ref.value, xe.value


def gemm_set_fwd_convert(on):
    """True: fp32 NCHW features go through the forward GEMM with in-kernel conversion where eligible; False (default): pack + GEMM
    (measured equal; env B200SEG_FWD_CONVERT=1 turns it on at load time)."""
    load().b200seg_gemm_set_fwd_convert(1 if on else 0)


def aspp_backward(grad_logits: torch.Tensor, Xp: torch.Tensor, WpT: torch.Tensor, rates: Sequence[int], N: int, h: int, w: int,
                  C: int, need_grad_x: bool = True, need_grad_w: bool = True, need_grad_b: bool = True, splits: int = 0):
    """Returns (grad_x fp32 NCHW | None, [grad_w]*R | None, [grad_b]*R | None)."""
    lib = load()
    grad_logits = _need(grad_logits.contiguous(), torch.float32, "grad_logits")
    Cin = WpT.shape[0]
    R = len(rates)
    dev = WpT.device
    if Xp is None and need_grad_w:
        raise B200SegError("aspp_backward: the weight gradient needs the packed features")
    if splits <= 0:
        splits = default_wgrad_splits(N * h * w, C, Cin, R)
    nbytes = lib.b200seg_aspp_backward_scratch_bytes(N, Cin, C, h, w, R, splits)
    scratch = _scratch("aspp_bwd", nbytes, dev)
    gx = torch.empty((N, Cin, h, w), dtype=torch.float32, device=dev) if need_grad_x else None
    gws = [torch.empty((C, Cin, 3, 3), dtype=torch.float32, device=dev) for _ in range(R)] if need_grad_w else None
    gbs = [torch.empty(C, dtype=torch.float32, device=dev) for _ in range(R)] if need_grad_b else None
    rates_arr = (c_int * R)(*[int(r) for r in rates])
    with _on_device(dev):
        _check(lib.b200seg_aspp_backward(grad_logits.data_ptr(), _ptr(Xp), WpT.data_ptr(), rates_arr, R, N, Cin, C, h, w,
                                         scratch.data_ptr(), nbytes, splits, _ptr(gx),
                                         _ptr_array(gws) if gws else None, _ptr_array(gbs) if gbs else None, _stream()))
    return gx, gws, gbs


def aspp_backward_packed(gOt: torch.Tensor, Xp: torch.Tensor, WpT: torch.Tensor, rates: Sequence[int], N: int, h: int, w: int,
                         C: int, need_grad_x: bool = True, need_grad_w: bool = True, splits: int = 0, nhwc_bf16: bool = False,
                         out_w: Optional[Sequence[torch.Tensor]] = None, weights_ready_event: Optional[torch.cuda.Event] = None):
    """Head backward from the packed bf16 gradient.  Returns (grad_x | None, [grad_w]*R | None); grad_x is fp32 NCHW, or with
    ``nhwc_bf16`` a bf16 channels_last tensor of logical shape [N,Cin,h,w] (the seam format, written directly by the GEMM).
    ``out_w``: R preallocated fp32 [C,Cin,3,3] buffers to write the weight gradients into (e.g. views of a flat DDP bucket);
    ``weights_ready_event`` is recorded on the current stream once they are complete, before the data-gradient GEMM."""
    lib = load()
    _need(gOt, torch.bfloat16, "gOt")
    Cin = WpT.shape[0]
    R = len(rates)
    dev = WpT.device
    if Xp is None and need_grad_w:
        raise B200SegError("aspp_backward_packed: the weight gradient needs the packed features")
    if splits <= 0:
        splits = default_wgrad_splits(N * h * w, C, Cin, R)
    nbytes = lib.b200seg_aspp_backward_scratch_bytes(N, Cin, C, h, w, R, splits)
    scratch = _scratch("aspp_bwd", nbytes, dev)
    gws = None
    if need_grad_w:
        if out_w is not None:
            gws = [_need(t, torch.float32, "out_w") for t in out_w]
            if len(gws) != R or any(tuple(t.shape) != (C, Cin, 3, 3) for t in gws):
                raise B200SegError("out_w: expected R contiguous fp32 [C,Cin,3,3] buffers")
        else:
            gws = [torch.empty((C, Cin, 3, 3), dtype=torch.float32, device=dev) for _ in range(R)]
    rates_arr = (c_int * R)(*[int(r) for r in rates])
    gx = gx_nhwc = None
    if need_grad_x:
        if nhwc_bf16:
            gx_nhwc = torch.empty((N, h, w, Cin), dtype=torch.bfloat16, device=dev)
        else:
            gx = torch.empty((N, Cin, h, w), dtype=torch.float32, device=dev)
    ev = None if weights_ready_event is None else weights_ready_event.cuda_event
    with _on_device(dev):
        _check(lib.b200seg_aspp_backward_packed_ex(gOt.data_ptr(), _ptr(Xp), WpT.data_ptr(), rates_arr, R, N, Cin, C, h, w,
                                                   scratch.data_ptr(), nbytes, splits, _ptr(gx), _ptr(gx_nhwc),
                                                   _ptr_array(gws) if gws else None, ev, _stream()))
    if gx_nhwc is not None:
        gx = gx_nhwc.permute(0, 3, 1, 2)
    return gx, gws


# --------------------------------------------------------------------------------------------
# K1 + K2 in one foreign call per direction (the fused train slice)
# --------------------------------------------------------------------------------------------
_head_loss_plans = {}


def _head_loss_plan(N, Cin, C, h, w, R, H, W, x_kind, rates):
    """(workspace bytes, scratch bytes, ctypes rate array) per shape -- computed once."""
    key = (N, Cin, C, h, w, R, H, W, x_kind, rates)
    plan = _head_loss_plans.get(key)
    if plan is None:
        lib = load()
        if len(_head_loss_plans) > 64:
            _head_loss_plans.clear()
        plan = (int(lib.b200seg_head_loss_workspace_bytes(N, Cin, C, h, w, R, H, W, x_kind)),
                int(lib.b200seg_head_loss_scratch_bytes(N, Cin, C, h, w, R)), (c_int * R)(*rates))
        _head_loss_plans[key] = plan
    return plan


def set_step_graphs(on: bool):
    """Graph replay of the one-call train entries (default on; env B200SEG_STEP_GRAPHS=0 turns it off at load time)."""
    load().b200seg_set_step_graphs(1 if on else 0)


def step_graph_stats():
    """(replays, captures) of the one-call train entries since the last set_step_graphs()."""
    a, b = ctypes.c_longlong(0), ctypes.c_longlong(0)
    load().b200seg_step_graph_stats(ctypes.byref(a), ctypes.byref(b))
    return a.value, b.value


def head_loss_forward(x: torch.Tensor, x_kind: int, shape, weights, biases, rates, labels: torch.Tensor, ignore_index: int,
                      inv_temperature: float, need_grad: bool):
    """pack -> head GEMM -> gather -> upsample + CE in ONE call.  ``x``: fp32 NCHW (x_kind 0) or bf16 pixel-major [N*h*w, Cin]
    (x_kind 1); ``shape`` = (N, Cin, h, w).  Returns (loss fp32 scalar tensor, logits fp32 [N,C,h,w], workspace) -- the workspace
    feeds head_loss_backward."""
    lib = load()
    N, Cin, h, w = shape
    R = len(rates)
    C = int(weights[0].shape[0])
    _need(x, torch.float32 if x_kind == 0 else torch.bfloat16, "features")
    for wt in weights:
        _need(wt, torch.float32, "conv weight")
        if tuple(wt.shape) != (C, Cin, 3, 3):
            raise B200SegError(f"conv weight shape {tuple(wt.shape)} != {(C, Cin, 3, 3)}")
    for b in biases:
        if b is not None:
            _need(b, torch.float32, "conv bias")
    lbytes = _need_label(labels, "labels")
    H, W = int(labels.shape[-2]), int(labels.shape[-1])
    if labels.numel() != N * H * W:
        raise B200SegError(f"labels shape {tuple(labels.shape)} does not match batch {N}")
    dev = x.device
    ws_bytes, sc_bytes, rates_arr = _head_loss_plan(N, Cin, C, h, w, R, H, W, x_kind, rates)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    logits = torch.empty((N, C, h, w), dtype=torch.float32, device=dev)
    loss = torch.empty((), dtype=torch.float32, device=dev)
    with _on_device(dev):
        scratch = _scratch("head_loss", sc_bytes, dev)
        _check(lib.b200seg_head_loss_forward(x.data_ptr(), x_kind, _ptr_array(weights), _ptr_array(biases), rates_arr, R, N, Cin, C, h, w,
                                             labels.data_ptr(), lbytes, H, W, ignore_index, inv_temperature, 1 if need_grad else 0,
                                             ws.data_ptr(), ws_bytes, scratch.data_ptr(), scratch.numel(), logits.data_ptr(),
                                             loss.data_ptr(), _stream()))
    return loss, logits, ws


def head_loss_backward(ws: torch.Tensor, x_bf16: Optional[torch.Tensor], x_kind: int, shape, C: int, rates, size, inv_temperature: float,
                       grad_loss: Optional[torch.Tensor], need_x: bool, need_w: bool, need_b: bool, nhwc_bf16: bool = False,
                       out_w=None, out_b=None, weights_ready_event=None):
    """Backward of head_loss_forward in ONE call.  Returns (grad_x | None, [grad_w]*R | None, [grad_b]*R | None); ``out_w`` /
    ``out_b``: preallocated destinations (views of a flat data-parallel bucket), ``weights_ready_event`` recorded once they are
    complete (before the data-gradient GEMM)."""
    lib = load()
    N, Cin, h, w = shape
    H, W = size
    R = len(rates)
    dev = ws.device
    _, sc_bytes, rates_arr = _head_loss_plan(N, Cin, C, h, w, R, H, W, x_kind, rates)
    if grad_loss is not None:
        grad_loss = _need(grad_loss.reshape(1), torch.float32, "grad_loss")
    gws = gbs = None
    if need_w:
        if out_w is not None:
            gws = [_need(t, torch.float32, "out_w") for t in out_w]
            if len(gws) != R or any(tuple(t.shape) != (C, Cin, 3, 3) for t in gws):
                raise B200SegError("out_w: expected R contiguous fp32 [C,Cin,3,3] buffers")
        else:
            gws = torch.empty((R, C, Cin, 3, 3), dtype=torch.float32, device=dev).unbind(0)
    if need_b:
        if out_b is not None:
            gbs = [_need(t, torch.float32, "out_b") for t in out_b]
            if len(gbs) != R or any(t.numel() != C for t in gbs):
                raise B200SegError("out_b: expected R contiguous fp32 [C] buffers")
        else:
            gbs = torch.empty((R, C), dtype=torch.float32, device=dev).unbind(0)
    gx = gx_nhwc = None
    if need_x:
        if nhwc_bf16:
            gx_nhwc = torch.empty((N, h, w, Cin), dtype=torch.bfloat16, device=dev)
        else:
            gx = torch.empty((N, Cin, h, w), dtype=torch.float32, device=dev)
    ev = None if weights_ready_event is None else weights_ready_event.cuda_event
    with _on_device(dev):
        scratch = _scratch("head_loss", sc_bytes, dev)
        _check(lib.b200seg_head_loss_backward(ws.data_ptr(), ws.numel(), _ptr(x_bf16), x_kind, rates_arr, R, N, Cin, C, h, w, H, W,
                                              inv_temperature, _ptr(grad_loss), scratch.data_ptr(), scratch.numel(), _ptr(gx),
                                              _ptr(gx_nhwc), _ptr_array(gws) if gws is not None else None,
                                              _ptr_array(gbs) if gbs is not None else None, ev, _stream()))
    if gx_nhwc is not None:
        gx = gx_nhwc.permute(0, 3, 1, 2)
    return gx, gws, gbs


# --------------------------------------------------------------------------------------------
# K6 in one foreign call per direction (the PixelDiscriminator conv stack, graph-replayed like the head entries)
# --------------------------------------------------------------------------------------------
def disc_forward(x: torch.Tensor, x_kind: int, shape, weights, biases, slope: float, packed=None):
    """cat(cls1, cls2)(LReLU(conv(LReLU(conv(x))))) in ONE call (weight pack, feature pack, three conv layers).  ``x``: fp32 NCHW
    (x_kind 0) or bf16 NHWC [N,h,w,Cin] (x_kind 1); ``shape`` = (N, Cin, h, w); ``weights`` = (w1, w2, wc1, wc2), ``biases`` =
    (b1, b2, bc1, bc2).  ``packed`` = ((Wf1,Wb1),(Wf2,Wb2),(Wf3,Wb3),b3) to reuse an existing pack (eval), None to pack inside the call.
    Returns (out fp32 [N,2C,h,w], Xp, A1, A2, packed)."""
    lib = load()
    N, Cin, h, w = shape
    w1, w2, wc1, wc2 = weights
    b1, b2, bc1, bc2 = biases
    ndf1, ndf2, C = int(w1.shape[0]), int(w2.shape[0]), int(wc1.shape[0])
    dev = x.device
    _need(x, torch.float32 if x_kind == 0 else torch.bfloat16, "features")
    for wt, shp in ((w1, (ndf1, Cin, 3, 3)), (w2, (ndf2, ndf1, 3, 3)), (wc1, (C, ndf2, 3, 3)), (wc2, (C, ndf2, 3, 3))):
        if tuple(_need(wt, torch.float32, "conv weight").shape) != shp:
            raise B200SegError(f"conv weight shape {tuple(wt.shape)}: expected {shp}")
    for b_ in biases:
        if b_ is not None:
            _need(b_, torch.float32, "conv bias")
    if Cin % 8 or ndf1 % 8 or ndf2 % 8:
        raise B200SegError("PixelDiscriminator: in_channels, ndf and ndf/2 must be multiples of 8")
    do_pack = packed is None
    if do_pack:
        bf = torch.bfloat16
        packed = ((torch.empty((9, ndf1, Cin), dtype=bf, device=dev), torch.empty((9, Cin, ndf1), dtype=bf, device=dev)),
                  (torch.empty((9, ndf2, ndf1), dtype=bf, device=dev), torch.empty((9, ndf1, ndf2), dtype=bf, device=dev)),
                  (torch.empty((9, 2 * C, ndf2), dtype=bf, device=dev), torch.empty((9, ndf2, _round8(2 * C)), dtype=bf, device=dev)),
                  torch.empty(2 * C, dtype=torch.float32, device=dev))
    (Wf1, Wb1), (Wf2, Wb2), (Wf3, Wb3), b3 = packed
    Xp = x if x_kind == 1 else torch.empty((N, h, w, Cin), dtype=torch.bfloat16, device=dev)
    A1 = torch.empty((N, h, w, ndf1), dtype=torch.bfloat16, device=dev)
    A2 = torch.empty((N, h, w, ndf2), dtype=torch.bfloat16, device=dev)
    out = torch.empty((N, 2 * C, h, w), dtype=torch.float32, device=dev)
    with _on_device(dev):
        _check(lib.b200seg_disc_forward(x.data_ptr(), x_kind, N, Cin, h, w, ndf1, ndf2, C, w1.data_ptr(), _ptr(b1), w2.data_ptr(), _ptr(b2),
                                        wc1.data_ptr(), _ptr(bc1), wc2.data_ptr(), _ptr(bc2), float(slope), 1 if do_pack else 0,
                                        Wf1.data_ptr(), Wb1.data_ptr(), Wf2.data_ptr(), Wb2.data_ptr(), Wf3.data_ptr(), Wb3.data_ptr(),
                                        b3.data_ptr(), None if x_kind == 1 else Xp.data_ptr(), A1.data_ptr(), A2.data_ptr(),
                                        out.data_ptr(), _stream()))
    return out, Xp, A1, A2, packed


def disc_backward(grad_out: torch.Tensor, Xp, A1, A2, Wb1, Wb2, Wb3, C: int, slope: float, need, x_bf16: bool):
    """Backward of disc_forward in ONE call.  ``need`` = (x, w1, b1, w2, b2, wc1, bc1, wc2, bc2) booleans.  Returns
    (gx | None, gw1, gb1, gw2, gb2, gwc1, gbc1, gwc2, gbc2) with None where not needed; gx is fp32 NCHW, or with ``x_bf16`` a bf16
    channels_last tensor of logical shape [N,Cin,h,w]."""
    lib = load()
    N, h, w, Cin = (int(v) for v in Xp.shape)
    ndf1, ndf2 = int(A1.shape[3]), int(A2.shape[3])
    dev = Xp.device
    grad_out = _need(grad_out, torch.float32, "grad_out")
    if tuple(grad_out.shape) != (N, 2 * C, h, w):
        raise B200SegError(f"disc_backward: grad_out shape {tuple(grad_out.shape)} != {(N, 2 * C, h, w)}")
    nx, nw1, nb1, nw2, nb2, nwc1, nbc1, nwc2, nbc2 = (bool(v) for v in need)
    f32, bf = torch.float32, torch.bfloat16
    need_l1 = nx or nw1 or nb1
    need_l2 = need_l1 or nw2 or nb2
    G3 = torch.empty((N, h, w, _round8(2 * C)), dtype=bf, device=dev)
    dZ2 = torch.empty((N, h, w, ndf2), dtype=bf, device=dev) if need_l2 else None
    dZ1 = torch.empty((N, h, w, ndf1), dtype=bf, device=dev) if need_l1 else None
    gw1 = torch.empty((ndf1, Cin, 3, 3), dtype=f32, device=dev) if nw1 else None
    gb1 = torch.empty(ndf1, dtype=f32, device=dev) if nb1 else None
    gw2 = torch.empty((ndf2, ndf1, 3, 3), dtype=f32, device=dev) if nw2 else None
    gb2 = torch.empty(ndf2, dtype=f32, device=dev) if nb2 else None
    gwc1 = torch.empty((C, ndf2, 3, 3), dtype=f32, device=dev) if nwc1 else None
    gwc2 = torch.empty((C, ndf2, 3, 3), dtype=f32, device=dev) if nwc2 else None
    gb3 = torch.empty(2 * C, dtype=f32, device=dev) if (nbc1 or nbc2) else None
    gx = gx_nhwc = None
    if nx:
        if x_bf16:
            gx_nhwc = torch.empty((N, h, w, Cin), dtype=bf, device=dev)
        else:
            gx = torch.empty((N, Cin, h, w), dtype=f32, device=dev)
    with _on_device(dev):
        nbytes = int(lib.b200seg_disc_backward_scratch_bytes(N, Cin, h, w, ndf1, ndf2, C))
        scratch = _scratch("disc_bwd", nbytes, dev)
        _check(lib.b200seg_disc_backward(grad_out.data_ptr(), Xp.data_ptr(), A1.data_ptr(), A2.data_ptr(), Wb1.data_ptr(), Wb2.data_ptr(),
                                         Wb3.data_ptr(), N, Cin, h, w, ndf1, ndf2, C, float(slope), G3.data_ptr(), _ptr(dZ2), _ptr(dZ1),
                                         scratch.data_ptr(), scratch.numel(), _ptr(gw1), _ptr(gb1), _ptr(gw2), _ptr(gb2), _ptr(gwc1),
                                         _ptr(gwc2), _ptr(gb3), _ptr(gx), _ptr(gx_nhwc), _stream()))
    if gx_nhwc is not None:
        gx = gx_nhwc.permute(0, 3, 1, 2)
    gbc1 = gb3[:C] if nbc1 else None
    gbc2 = gb3[C:] if nbc2 else None
    return gx, gw1, gb1, gw2, gb2, gwc1, gbc1, gwc2, gbc2


# --------------------------------------------------------------------------------------------
# K6  3x3 conv layers as tcgen05 implicit GEMMs (PixelDiscriminator stack), bf16 NHWC activations
# --------------------------------------------------------------------------------------------
def _round8(v: int) -> int:
    return (int(v) + 7) // 8 * 8


def conv3x3_pack_weights(weights: Sequence[torch.Tensor]):
    """[Co_i,Ci,3,3] fp32 tensors (concatenated along Co) -> (Wf bf16 [9,Co,Ci], Wb bf16 [9,Ci,round8(Co)])."""
    lib = load()
    Ci = weights[0].shape[1]
    for wt in weights:
        _need(wt, torch.float32, "conv weight")
        if wt.dim() != 4 or tuple(wt.shape[1:]) != (Ci, 3, 3):
            raise B200SegError(f"conv weight shape {tuple(wt.shape)}: expected [Co,{Ci},3,3]")
    if Ci % 8 != 0:
        raise B200SegError(f"conv3x3: in_channels={Ci} must be a multiple of 8")
    parts = [int(wt.shape[0]) for wt in weights]
    Co = sum(parts)
    dev = weights[0].device
    Wf = torch.empty((9, Co, Ci), dtype=torch.bfloat16, device=dev)
    Wb = torch.empty((9, Ci, _round8(Co)), dtype=torch.bfloat16, device=dev)       # padding columns are zero-filled by the kernel
    with _on_device(dev):
        _check(lib.b200seg_conv3x3_pack_weights(_ptr_array(weights), (c_int * len(parts))(*parts), len(parts), Ci, Wf.data_ptr(),
                                                Wb.data_ptr(), Wb.shape[2], _stream()))
    return Wf, Wb


def conv3x3_pack_weights_stack(layers: Sequence[Sequence[torch.Tensor]], bias_parts: Sequence[Optional[torch.Tensor]] = (),
                               bias_lens: Sequence[int] = ()):
    """Every layer of a conv stack in ONE launch: ``layers[l]`` = the [Co_i,Ci_l,3,3] fp32 tensors concatenated along Co for layer
    l.  Returns ([(Wf_l, Wb_l)], bias) with bias = the concatenation of ``bias_parts`` (None = zeros of ``bias_lens[i]``)."""
    lib = load()
    flat, parts, ppl, cis, Wfs, Wbs, pitches = [], [], [], [], [], [], []
    dev = layers[0][0].device
    for ws in layers:
        Ci = int(ws[0].shape[1])
        for wt in ws:
            _need(wt, torch.float32, "conv weight")
            if wt.dim() != 4 or tuple(wt.shape[1:]) != (Ci, 3, 3) or wt.device != dev:
                raise B200SegError(f"conv weight shape {tuple(wt.shape)}: expected [Co,{Ci},3,3] on {dev}")
        if Ci % 8 != 0:
            raise B200SegError(f"conv3x3: in_channels={Ci} must be a multiple of 8")
        Co = sum(int(wt.shape[0]) for wt in ws)
        flat += list(ws)
        parts += [int(wt.shape[0]) for wt in ws]
        ppl.append(len(ws))
        cis.append(Ci)
        Wfs.append(torch.empty((9, Co, Ci), dtype=torch.bfloat16, device=dev))
        Wbs.append(torch.empty((9, Ci, _round8(Co)), dtype=torch.bfloat16, device=dev))
        pitches.append(_round8(Co))
    bias = None
    if bias_lens:
        for b_, n_ in zip(bias_parts, bias_lens):
            if b_ is not None and (_need(b_, torch.float32, "bias").numel() != n_):
                raise B200SegError("conv3x3_pack_weights_stack: bias length mismatch")
        bias = torch.empty(int(sum(bias_lens)), dtype=torch.float32, device=dev)
    ia = lambda v: (c_int * len(v))(*[int(x) for x in v])  # noqa: E731
    with _on_device(dev):
        _check(lib.b200seg_conv3x3_pack_weights_stack(len(layers), _ptr_array(flat), ia(parts), ia(ppl), ia(cis), _ptr_array(Wfs),
                                                      _ptr_array(Wbs), ia(pitches), _ptr_array(list(bias_parts)) if bias_lens else None,
                                                      ia(bias_lens) if bias_lens else None, len(bias_lens), _ptr(bias), _stream()))
    return list(zip(Wfs, Wbs)), bias


def _need_nhwc(t: torch.Tensor, name: str):
    _need(t, torch.bfloat16, name)
    if t.dim() != 4 or t.shape[3] % 8 != 0:
        raise B200SegError(f"{name}: expected bf16 NHWC [N,h,w,C] with C a multiple of 8, got {tuple(t.shape)}")
    return t.shape


def conv3x3_forward(act: torch.Tensor, Wf: torch.Tensor, bias: Optional[torch.Tensor], lrelu_slope: Optional[float] = None,
                    dilation: int = 1, out_f32_nchw: bool = False) -> torch.Tensor:
    """[LeakyReLU](conv3x3(act) + bias) with padding == dilation.  act bf16 NHWC [N,h,w,Ci]; returns bf16 NHWC [N,h,w,round8(Co)]
    (requires Co % 8 == 0) or, with ``out_f32_nchw``, fp32 NCHW [N,Co,h,w]."""
    lib = load()
    N, h, w, pitch = _need_nhwc(act, "act")
    _need(Wf, torch.bfloat16, "Wf")
    Co, Ci = int(Wf.shape[1]), int(Wf.shape[2])
    if Ci != pitch:
        raise B200SegError(f"conv3x3_forward: activations have {pitch} channels, weights expect {Ci}")
    if bias is not None:
        _need(bias, torch.float32, "bias")
    out_b = out_f = None
    if out_f32_nchw:
        out_f = torch.empty((N, Co, h, w), dtype=torch.float32, device=act.device)
    else:
        if Co % 8 != 0:
            raise B200SegError(f"conv3x3_forward: bf16 NHWC output needs out_channels={Co} to be a multiple of 8")
        out_b = torch.empty((N, h, w, Co), dtype=torch.bfloat16, device=act.device)
    with _on_device(act.device):
        _check(lib.b200seg_conv3x3_forward(act.data_ptr(), N, h, w, Ci, pitch, Wf.data_ptr(), Co, int(dilation), _ptr(bias),
                                           0 if lrelu_slope is None else 1, 0.0 if lrelu_slope is None else float(lrelu_slope),
                                           _ptr(out_b), Co, _ptr(out_f), _stream()))
    return out_f if out_f32_nchw else out_b


def conv3x3_dgrad(g: torch.Tensor, Wb: torch.Tensor, mask: Optional[torch.Tensor] = None, slope: float = 0.2, dilation: int = 1,
                  out_f32_nchw: bool = False, want_colsum: bool = False):
    """Data gradient of conv3x3 (padding == dilation): g bf16 NHWC [N,h,w,round8(Co)], Wb bf16 [9,Ci,round8(Co)].  ``mask`` (bf16
    NHWC [N,h,w,Ci], the saved LeakyReLU output of the layer below) fuses the activation's backward into the epilogue.
    ``want_colsum`` (bf16 NHWC output only) returns (gradient, fp32 [Ci] per-channel sums of the gradient) -- the bias gradient of
    the layer below, accumulated in the same epilogue."""
    lib = load()
    N, h, w, gp = _need_nhwc(g, "g")
    _need(Wb, torch.bfloat16, "Wb")
    Ci, Cg = int(Wb.shape[1]), int(Wb.shape[2])
    if Cg != gp:
        raise B200SegError(f"conv3x3_dgrad: gradient has {gp} channels, Wb expects {Cg}")
    out_b = out_f = None
    if out_f32_nchw:
        if mask is not None:
            raise B200SegError("conv3x3_dgrad: the fused activation mask needs the bf16 NHWC output")
        out_f = torch.empty((N, Ci, h, w), dtype=torch.float32, device=g.device)
    else:
        if Ci % 8 != 0:
            raise B200SegError(f"conv3x3_dgrad: bf16 NHWC output needs in_channels={Ci} to be a multiple of 8")
        out_b = torch.empty((N, h, w, Ci), dtype=torch.bfloat16, device=g.device)
        if mask is not None and tuple(_need_nhwc(mask, "mask")) != (N, h, w, Ci):
            raise B200SegError(f"conv3x3_dgrad: mask shape {tuple(mask.shape)} != {(N, h, w, Ci)}")
    if want_colsum:
        if out_f32_nchw:
            raise B200SegError("conv3x3_dgrad: the fused column sums need the bf16 NHWC output")
        nbytes = lib.b200seg_conv3x3_dgrad_colsum_scratch_bytes(N, h, w, Ci)
        scratch = _scratch("dgrad_colsum", nbytes, g.device)
        colsum = torch.empty(Ci, dtype=torch.float32, device=g.device)
        with _on_device(g.device):
            _check(lib.b200seg_conv3x3_dgrad_colsum(g.data_ptr(), N, h, w, Cg, gp, Wb.data_ptr(), Ci, int(dilation), _ptr(mask),
                                                    float(slope), out_b.data_ptr(), Ci, scratch.data_ptr(), nbytes,
                                                    colsum.data_ptr(), _stream()))
        return out_b, colsum
    with _on_device(g.device):
        _check(lib.b200seg_conv3x3_dgrad(g.data_ptr(), N, h, w, Cg, gp, Wb.data_ptr(), Ci, int(dilation), _ptr(mask), float(slope),
                                         _ptr(out_b), Ci, _ptr(out_f), _stream()))
    return out_f if out_f32_nchw else out_b


def conv3x3_wgrad(g: torch.Tensor, x: torch.Tensor, parts: Sequence[int], dilation: int = 1, splits: int = 0,
                  out: Optional[Sequence[Optional[torch.Tensor]]] = None):
    """Weight gradients [parts[i],Ci,3,3] fp32 from the bf16 NHWC output gradient g [N,h,w,round8(sum parts)] and input x."""
    lib = load()
    N, h, w, gp = _need_nhwc(g, "g")
    if tuple(_need_nhwc(x, "x"))[:3] != (N, h, w):
        raise B200SegError("conv3x3_wgrad: g and x must share [N,h,w]")
    Ci = int(x.shape[3])
    Co = int(sum(parts))
    if _round8(Co) != gp:
        raise B200SegError(f"conv3x3_wgrad: gradient has {gp} channels, parts sum to {Co}")
    nbytes = lib.b200seg_conv3x3_wgrad_scratch_bytes(N, h, w, Co, Ci, int(splits))
    scratch = _scratch("conv_wgrad", nbytes, g.device)
    if out is None:
        out = [torch.empty((int(pc), Ci, 3, 3), dtype=torch.float32, device=g.device) for pc in parts]
    for t, pc in zip(out, parts):
        if t is not None and (tuple(_need(t, torch.float32, "grad_w").shape) != (int(pc), Ci, 3, 3)):
            raise B200SegError("conv3x3_wgrad: bad output buffer shape")
    with _on_device(g.device):
        _check(lib.b200seg_conv3x3_wgrad(g.data_ptr(), Co, gp, x.data_ptr(), Ci, Ci, N, h, w, int(dilation), int(splits),
                                         scratch.data_ptr(), nbytes, _ptr_array(out), (c_int * len(parts))(*[int(v) for v in parts]),
                                         len(parts), _stream()))
    return list(out)


def nchw_to_nhwc_bf16(src: torch.Tensor, pitch: Optional[int] = None) -> torch.Tensor:
    """fp32 NCHW [N,C,h,w] -> bf16 NHWC [N,h,w,pitch] (pitch = round8(C) by default; channels >= C are zero)."""
    lib = load()
    _need(src, torch.float32, "src")
    N, C, h, w = src.shape
    pitch = _round8(C) if pitch is None else int(pitch)
    dst = torch.empty((N, h, w, pitch), dtype=torch.bfloat16, device=src.device)
    with _on_device(src.device):
        _check(lib.b200seg_nchw_to_nhwc_bf16(src.data_ptr(), N, C, h * w, dst.data_ptr(), pitch, _stream()))
    return dst


def _need_channels_last_bf16(t: torch.Tensor, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor, got {type(t)}")
    if not t.is_cuda:
        raise B200SegError(f"{name}: expected a CUDA tensor (b200seg has no CPU fallback), got device {t.device}")
    if t.dtype != torch.bfloat16 or t.dim() != 4 or not t.is_contiguous(memory_format=torch.channels_last):
        raise B200SegError(f"{name}: expected a bf16 channels_last contiguous [N,C,h,w] tensor")
    return t


def _need_channel_vector(t: torch.Tensor, C: int, name: str) -> torch.Tensor:
    _need(t, torch.float32, name)
    if t.numel() != C:
        raise B200SegError(f"{name}: expected {C} values, got {t.numel()}")
    return t


def seam_tail_forward(c: torch.Tensor, identity: torch.Tensor, scale: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """bf16 channels_last y = bf16_rn(relu((c * scale + bias) + identity)) from fp32 NCHW c / identity (the last Bottleneck's
    bn3 + residual + relu, resnet.py:106-113, with the cast the head's seam format takes); bit-identical to the stock fp32
    result .to(torch.bfloat16).  C % 8 == 0."""
    lib = load()
    _need(c, torch.float32, "c")
    _need(identity, torch.float32, "identity")
    if c.dim() != 4 or identity.shape != c.shape:
        raise B200SegError(f"seam_tail_forward: c {tuple(c.shape)} and identity {tuple(identity.shape)} must be equal [N,C,h,w]")
    N, C, h, w = c.shape
    _need_channel_vector(scale, C, "scale")
    _need_channel_vector(bias, C, "bias")
    y = torch.empty((N, C, h, w), dtype=torch.bfloat16, device=c.device, memory_format=torch.channels_last)
    with _on_device(c.device):
        _check(lib.b200seg_seam_tail_forward(c.data_ptr(), identity.data_ptr(), scale.data_ptr(), bias.data_ptr(), N, C, h * w,
                                             y.data_ptr(), _stream()))
    return y


def seam_tail_backward(dy: torch.Tensor, y: torch.Tensor, scale: torch.Tensor, need_c: bool = True, need_identity: bool = True):
    """(dc, didentity), fp32 NCHW: g = dy * (y > 0), dc = g * scale, didentity = g; dy / y bf16 channels_last.  An output that is
    not needed is None (and not written)."""
    lib = load()
    _need_channels_last_bf16(dy, "dy")
    _need_channels_last_bf16(y, "y")
    if dy.shape != y.shape:
        raise B200SegError(f"seam_tail_backward: dy {tuple(dy.shape)} and y {tuple(y.shape)} differ")
    N, C, h, w = y.shape
    _need_channel_vector(scale, C, "scale")
    dc = torch.empty((N, C, h, w), dtype=torch.float32, device=y.device) if need_c else None
    di = torch.empty((N, C, h, w), dtype=torch.float32, device=y.device) if need_identity else None
    if dc is None and di is None:
        return None, None
    with _on_device(y.device):
        _check(lib.b200seg_seam_tail_backward(dy.data_ptr(), y.data_ptr(), scale.data_ptr(), N, C, h * w, _ptr(dc), _ptr(di), _stream()))
    return dc, di


def nhwc_bf16_colsum(g: torch.Tensor, C: Optional[int] = None) -> torch.Tensor:
    """out[c] = sum over pixels of g[..., c] (bias gradient), fp32 [C], deterministic."""
    lib = load()
    N, h, w, pitch = _need_nhwc(g, "g")
    C = pitch if C is None else int(C)
    nbytes = lib.b200seg_nhwc_colsum_scratch_bytes(pitch)
    scratch = _scratch("colsum", nbytes, g.device)
    out = torch.empty(C, dtype=torch.float32, device=g.device)
    with _on_device(g.device):
        _check(lib.b200seg_nhwc_bf16_colsum(g.data_ptr(), N * h * w, C, pitch, scratch.data_ptr(), out.data_ptr(), _stream()))
    return out


def default_wgrad_splits(P: int, C: int, Cin: int, R: int) -> int:
    """Split-K factor for the weight-gradient GEMM.  It runs as CTA pairs (two M-tiles per pair, 74 pairs): take the smallest
    factor >= 4 whose pair-unit count fills whole rounds of the 74 pairs best (NJ = 640, Cin = 2048: 3 x 8 x 6 = 144 units = 2 rounds
    at 97 %)."""
    NJ = aspp_packed_rows(C, R)
    pairs_m = ((NJ + 127) // 128 + 1) // 2
    tiles = pairs_m * ((Cin + 255) // 256)
    kb = (P + 63) // 64
    workers = 74
    best, best_eff = 1, -1.0
    for s in range(1, 17):
        if s > kb:
            break
        units = tiles * s
        eff = units / (((units + workers - 1) // workers) * workers)
        if s >= 4 and eff > best_eff + 1e-9:
            best, best_eff = s, eff
    return int(best if best_eff > 0 else max(1, min(kb, 4)))


def gemm_selftest(M, N, K, a_mn=False, b_mn=False, splits=1, col_hw=0, share=0):
    lib = load()
    err, ref = ctypes.c_double(0), ctypes.c_double(0)
    _check(lib.b200seg_gemm_selftest(M, N, K, int(a_mn), int(b_mn), splits, col_hw, int(share), ctypes.byref(err), ctypes.byref(ref)))
    return err.value, ref.value


def gemm_set_dgrad_mode(mode: int):
    """fp32 NCHW data gradient of the head: 0 = channel-major GEMM with the shared-memory transpose epilogue, 1 (default) = pixel-major
    CTA pairs storing straight from registers (seven ring stages)."""
    load().b200seg_gemm_set_dgrad_mode(int(mode))


def gemm_set_fwd_mode(mode: int):
    """Head forward GEMM: 0 = channel-major, 1 (default) = pixel-major with the ragged last N-tile at half MMA width."""
    load().b200seg_gemm_set_fwd_mode(int(mode))


def gemm_set_narrow_tiles(on):
    """Head forward GEMM: True (default) = 256 / 224 / 192-column tiles chosen per problem against wave quantisation."""
    load().b200seg_gemm_set_narrow_tiles(1 if on else 0)


def conv_set_pair(on):
    """K6: True (default) = CTA pairs on one tcgen05.mma.cta_group::2 where a layer has two M-tiles; False = one CTA per tile."""
    load().b200seg_conv_set_pair(1 if on else 0)


def gemm_set_sharing(mode):
    """0 / False: no multicast; 1 / True: 2-CTA pairs (default); 2: 2 x 2 clusters multicasting both operands (slower: kept for A/B)."""
    load().b200seg_gemm_set_sharing(int(mode))


PROFILE_TAGS = {"head_fwd_gemm": 0, "head_dgrad_gemm": 1, "head_wgrad_gemm": 2, "pack_features": 3, "head_gather": 4,
                "grad_im2col": 5, "upsample_ce_main": 6, "eval_argmax_confusion": 7, "soft_ce_fwd": 8, "soft_ce_bwd": 9,
                "wgrad_reduce": 10, "fada_softce_main": 11, "conv3x3_fwd": 12, "conv3x3_dgrad": 13, "conv3x3_wgrad": 14, "tta": 15}


def launch_count() -> int:
    return int(load().b200seg_launch_count())


def gemm_set_overlap_sms(n: int):
    load().b200seg_gemm_set_overlap_sms(int(n))


def profile_enable(on: bool):
    load().b200seg_profile_enable(1 if on else 0)


def profile_read():
    """{kernel name: (total_ms, launches)} accumulated since profile_enable(True)."""
    lib = load()
    out = {}
    for name, tag in PROFILE_TAGS.items():
        ms, n = ctypes.c_double(0), c_int(0)
        _check(lib.b200seg_profile_read(tag, ctypes.byref(ms), ctypes.byref(n)))
        if n.value:
            out[name] = (ms.value, n.value)
    return out
