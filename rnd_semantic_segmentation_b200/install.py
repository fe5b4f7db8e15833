"""Patch the B200 hot path into an importable copy of the reference tree.

    import rnd_semantic_segmentation_b200 as b200seg
    b200seg.install()          # before train_src.py / train_adv.py / test.py build their models

After this, ``core.models.build.build_classifier`` / ``build_adversarial_discriminator`` and
``core.utils.utility.{soft_label_cross_entropy,inference,multi_scale_inference,intersectionAndUnionGPU,confusion_matrix,
AverageMeter,get_color_palette}`` and ``core.utils.adapt_lr.adjust_learning_rate`` resolve to this package's implementations; the
scripts themselves stay unmodified (INTEGRATION.md).  ``install(optimizers=True)`` additionally makes the trainers'
``torch.optim.SGD`` / ``torch.optim.Adam`` constructions (aspp_trainer.py:25-26, fada_adapter.py:24) build FusedSGD / FusedAdam for
parameter sets that live on a CUDA device (everything else keeps the stock classes).  ``install(seam=True)`` additionally wraps
``core.models.build.build_feature_extractor`` (same signature) so that the backbone it returns emits the head's seam format, bf16
channels_last, from its last Bottleneck (seam.fuse_backbone_tail; INTEGRATION.md "Seam format").
"""
from __future__ import annotations

import importlib
import sys

import torch

from . import build as _build
from . import optim as _optim
from . import seam as _seam
from . import utility as _utility

_BUILD_NAMES = ("build_classifier", "build_adversarial_discriminator")
_UTIL_NAMES = ("soft_label_cross_entropy", "inference", "multi_scale_inference", "intersectionAndUnionGPU", "confusion_matrix",
               "AverageMeter", "get_color_palette")
_LR_NAMES = ("adjust_learning_rate",)
_stock_optimizers = {}


def _optimizer_factory(stock, fused):
    """A CLASS that stands in for ``torch.optim.SGD`` / ``torch.optim.Adam``: constructing it builds the fused subclass for
    all-CUDA fp32 parameter sets and the stock class otherwise (the backbone's optimizer_fea is one of those calls too; it takes
    the fused path just the same when it is on the GPU).  It stays a type: ``isinstance(opt, torch.optim.SGD)`` and
    ``issubclass`` answer as for the stock class, and ``class X(torch.optim.SGD)`` keeps working (a subclass constructs itself
    normally, on the stock implementation)."""

    class _Meta(type(stock)):
        def __instancecheck__(cls, obj):
            return isinstance(obj, stock) if cls is dispatch_holder[0] else type.__instancecheck__(cls, obj)

        def __subclasscheck__(cls, sub):
            return issubclass(sub, stock) if cls is dispatch_holder[0] else type.__subclasscheck__(cls, sub)

    dispatch_holder = [None]

    def __new__(cls, params=None, *args, **kwargs):
        if cls is not dispatch_holder[0]:                      # a user subclass: ordinary construction
            return stock.__new__(cls)
        params = list(params)
        flat = [p for g in params for p in g["params"]] if params and isinstance(params[0], dict) else params
        if flat and all(isinstance(p, torch.Tensor) and p.is_cuda and p.dtype == torch.float32 for p in flat):
            return fused(params, *args, **kwargs)
        return stock(params, *args, **kwargs)                  # neither result is an instance of `cls`: no second __init__

    dispatch = _Meta(stock.__name__, (stock,), {"__new__": __new__, "__wrapped__": stock, "__module__": stock.__module__,
                                                "__doc__": stock.__doc__})
    dispatch_holder[0] = dispatch
    return dispatch


def install_optimizers():
    """torch.optim.SGD / torch.optim.Adam -> factories that build FusedSGD / FusedAdam for CUDA fp32 parameters."""
    if not _stock_optimizers:
        _stock_optimizers.update(SGD=torch.optim.SGD, Adam=torch.optim.Adam)
        torch.optim.SGD = _optimizer_factory(_stock_optimizers["SGD"], _optim.FusedSGD)
        torch.optim.Adam = _optimizer_factory(_stock_optimizers["Adam"], _optim.FusedAdam)
    return ["torch.optim.SGD", "torch.optim.Adam"]


def uninstall_optimizers():
    if _stock_optimizers:
        torch.optim.SGD, torch.optim.Adam = _stock_optimizers.pop("SGD"), _stock_optimizers.pop("Adam")


def _install_seam(patched):
    """core.models(.build).build_feature_extractor -> the same factory with fuse_backbone_tail applied to its result, also in
    modules that imported the name before."""
    wrapped = {}                     # id(stock function) -> wrapper (core.models re-exports core.models.build's function)
    for modname in ("core.models.build", "core.models"):
        mod = sys.modules.get(modname)
        stock = getattr(mod, "build_feature_extractor", None) if mod is not None else None
        if stock is None:
            continue
        fn = wrapped.setdefault(id(stock), _seam.wrap_feature_extractor_factory(stock))
        wrapped[id(fn)] = fn
        setattr(mod, "build_feature_extractor", fn)
        patched.append(f"{modname}.build_feature_extractor")
    for mod in list(sys.modules.values()):
        name = getattr(mod, "__name__", "")
        if not name.startswith("core.") or name in ("core.models.build", "core.models"):
            continue
        fn = getattr(mod, "__dict__", {}).get("build_feature_extractor")
        if fn is not None and id(fn) in wrapped:
            setattr(mod, "build_feature_extractor", wrapped[id(fn)])
            patched.append(f"{name}.build_feature_extractor")


def install(strict: bool = False, optimizers: bool = False, seam: bool = False):
    """Returns the list of 'module.attr' names that were patched.  ``seam=True``: the reference's build_feature_extractor returns
    a backbone whose last Bottleneck emits bf16 channels_last features (seam.fuse_backbone_tail)."""
    patched = install_optimizers() if optimizers else []
    targets = (("core.models.build", _build, _BUILD_NAMES), ("core.models", _build, _BUILD_NAMES),
               ("core.utils.utility", _utility, _UTIL_NAMES), ("core.utils.adapt_lr", _optim, _LR_NAMES))
    for modname, src, names in targets:
        mod = sys.modules.get(modname)
        if mod is None:
            try:
                mod = importlib.import_module(modname)
            except Exception:
                if strict:
                    raise
                continue
        for n in names:
            setattr(mod, n, getattr(src, n))
            patched.append(f"{modname}.{n}")
    # modules that did `from core.utils.utility import X` / `from core.models import build_*` before install()
    for mod in list(sys.modules.values()):
        name = getattr(mod, "__name__", "")
        if not name.startswith("core.") or name in ("core.models.build", "core.models", "core.utils.utility", "core.utils.adapt_lr"):
            continue
        for src, names in ((_build, _BUILD_NAMES), (_utility, _UTIL_NAMES), (_optim, _LR_NAMES)):
            for n in names:
                if n in getattr(mod, "__dict__", {}):
                    setattr(mod, n, getattr(src, n))
                    patched.append(f"{name}.{n}")
    if seam:
        _install_seam(patched)
    return patched
