"""Factory API -- the plug-in seam of the reference, core/models/build.py:13-52, signatures unchanged.

``cfg`` is duck-typed: only ``cfg.MODEL.NAME`` ("<model>_<backbone>") and ``cfg.MODEL.NUM_CLASSES``
are read, exactly as the reference does.
"""
from __future__ import annotations

import functools

from .classifier import ASPP_Classifier_V2
from .discriminator import PixelDiscriminator

__all__ = ["build_feature_extractor", "build_classifier", "build_adversarial_discriminator", "wrap_discriminator_factory"]

_ASPP_RATES = [6, 12, 18, 24]


def build_feature_extractor(cfg):
    """build.py:13-21.  The backbone is outside this package's scope (SURVEY.md section 2 row 5): it is delegated to
    the reference's own ``core.models.feature_extractor`` when that tree is importable."""
    _, backbone_name = cfg.MODEL.NAME.split('_')
    if not (backbone_name.startswith('resnet') or backbone_name.startswith('vgg')):
        raise NotImplementedError
    try:
        from core.models import feature_extractor as ref_fe  # the reference tree, if on sys.path
    except Exception as e:  # pragma: no cover - depends on the host environment
        raise ImportError("build_feature_extractor delegates to the reference's backbone "
                          "(core.models.feature_extractor), which is not importable here") from e
    fn = ref_fe.resnet_feature_extractor if backbone_name.startswith('resnet') else ref_fe.vgg_feature_extractor
    return fn(backbone_name, pretrained_weights=cfg.MODEL.WEIGHTS, aux=False, pretrained_backbone=True,
              freeze_bn=cfg.MODEL.FREEZE_BN)


def build_classifier(cfg):
    """build.py:23-31."""
    _, backbone_name = cfg.MODEL.NAME.split('_')
    if backbone_name.startswith('vgg'):
        return ASPP_Classifier_V2(1024, _ASPP_RATES, _ASPP_RATES, cfg.MODEL.NUM_CLASSES)
    if backbone_name.startswith('resnet'):
        return ASPP_Classifier_V2(2048, _ASPP_RATES, _ASPP_RATES, cfg.MODEL.NUM_CLASSES)
    raise NotImplementedError


def build_adversarial_discriminator(cfg, num_features=None, mid_nc=256):
    """build.py:33-52."""
    _, backbone_name = cfg.MODEL.NAME.split('_')
    defaults = (('vgg', 1024), ('resnet', 2048), ('efficientnet', 1408), ('hardnet', 1024))
    for prefix, feats in defaults:
        if backbone_name.startswith(prefix):
            if num_features is None:
                num_features = feats
            return PixelDiscriminator(num_features, mid_nc, num_classes=cfg.MODEL.NUM_CLASSES)
    raise NotImplementedError


def wrap_discriminator_factory(stock, tf32: bool = False):
    """``build_adversarial_discriminator`` with the same signature whose PixelDiscriminator results get ``tf32`` set
    (install(disc_tf32=True)).  Wrapping a wrapper returns it with its flag set to the new value."""
    if getattr(stock, "_b200seg_disc", False):
        stock._b200seg_disc_tf32 = bool(tf32)
        return stock

    @functools.wraps(stock)
    def build_adversarial_discriminator(*args, **kwargs):
        D = stock(*args, **kwargs)
        if isinstance(D, PixelDiscriminator):
            D.tf32 = build_adversarial_discriminator._b200seg_disc_tf32
        return D

    build_adversarial_discriminator._b200seg_disc = True
    build_adversarial_discriminator._b200seg_disc_tf32 = bool(tf32)
    return build_adversarial_discriminator
