"""rnd_semantic_segmentation_b200 -- B200-native (sm_100a) hot path of taintpro98/rnd-semantic-segmentation.

Drop-in for ONE path: DeepLabV2 ASPP classifier head -> align-corners upsample -> (hard / soft-label)
cross-entropy fwd/bwd -> PixelDiscriminator loss tail -> argmax + confusion matrix / mIoU.
Host code is Python/PyTorch (memory, streams, autograd, torch.distributed); the arithmetic is hand-written
CUDA behind the C ABI in include/b200seg.h (libb200seg.so).  No CPU fallback.
"""
from .build import build_adversarial_discriminator, build_classifier, build_feature_extractor
from .classifier import ASPP_Classifier_V2
from .discriminator import PixelDiscriminator
from .install import install
from .ops import (aspp_head, aspp_head_loss, clear_feature_pack_cache, fada_soft_label_loss, seam_tail, set_feature_pack_cache, soft_label_cross_entropy, upsample_bilinear_align_corners, upsample_cross_entropy)
from .utility import (AverageMeter, BatchedEvaluator, confusion_matrix, get_color_palette, inference, intersectionAndUnion, intersectionAndUnionGPU,
                      iutr_from_confusion, multi_scale_inference, pseudo_label_map, save_pseudo_label, segmentation_eval_step)
from .optim import FusedAdam, FusedSGD, adjust_learning_rate
from .seam import fuse_backbone_tail, unfuse_backbone_tail

__all__ = [
    "build_feature_extractor", "build_classifier", "build_adversarial_discriminator",
    "ASPP_Classifier_V2", "PixelDiscriminator", "install",
    "aspp_head", "aspp_head_loss", "fada_soft_label_loss", "upsample_bilinear_align_corners", "upsample_cross_entropy", "soft_label_cross_entropy",
    "inference", "multi_scale_inference", "pseudo_label_map", "get_color_palette", "save_pseudo_label", "FusedSGD", "FusedAdam", "adjust_learning_rate", "intersectionAndUnion", "intersectionAndUnionGPU", "confusion_matrix", "AverageMeter",
    "segmentation_eval_step", "iutr_from_confusion", "BatchedEvaluator", "set_feature_pack_cache", "clear_feature_pack_cache",
    "fuse_backbone_tail", "unfuse_backbone_tail", "seam_tail",
]
