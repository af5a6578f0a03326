"""ucd_b200 - B200-native (sm_100a) implementation of UCD's distillation-loss hot path.

Drop-in loss modules with the reference's names and signatures; see ucd_b200/losses.py,
include/ucd_b200.h (the C ABI) and INTEGRATION.md.
"""
from .losses import (ContrastPack, FusedUnbiasedLosses, JointProb, KnowledgeDistillationLoss,  # noqa: F401
                     MaskCrossEntropy, MaskKnowledgeDistillationLoss, PixelConLoss, PixelConLossV2,
                     PixelContrastiveDistillation, SupConLoss, UnbiasedCrossEntropy, UnbiasedKnowledgeDistillationLoss,
                     interpolate_bilinear, pre_contractive_pixel, pre_contrastive_pixel, predict_bilinear)
from ._lib import enable_nvtx  # noqa: F401

__all__ = ["PixelConLossV2", "UnbiasedCrossEntropy", "UnbiasedKnowledgeDistillationLoss", "pre_contrastive_pixel",
           "pre_contractive_pixel", "interpolate_bilinear", "JointProb", "ContrastPack", "FusedUnbiasedLosses",
           "PixelContrastiveDistillation", "enable_nvtx", "KnowledgeDistillationLoss", "MaskKnowledgeDistillationLoss", "MaskCrossEntropy", "PixelConLoss", "SupConLoss", "predict_bilinear"]
