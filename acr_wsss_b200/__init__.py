"""acr_wsss_b200 -- B200-native (sm_100a) implementation of the ACR_WSSS all-pairs attention-affinity hot path.

Public surface (mirrors the reference's names for this path):
    ACR, Attention, VisionTransformer          (model.py    <- DPT/ACR.py, models/vision_transformer.py)
    acr_consistency_loss, acr_total_loss       (losses.py   <- train_acr.py:140-168)
    affinity_refine, infer_cam_image/_batch    (cam.py      <- infer_cam.py:145-215)
    save_cam_dict, pseudo_label, label_iou     (cam.py      <- infer_cam.py:227-228, evaluation.py:28-67)
    crf_inference, crf_with_alpha(_batch)      (cam.py      <- tool/imutils.py crf_inference, myTool.py _crf_with_alpha)
    PAMR                                       (pamr.py     <- pamr.py)
    bilateralfilter_batch                      (bilateralfilter.py <- wrapper/bilateralfilter)
    GpuAugment, Prefetcher, augment_params     (data.py     <- myTool.py:1158-1199 get_data_from_chunk_v2)
All compute goes through libacr_b200.so (csrc/, C ABI in include/acr_b200.h); there is no CPU fallback.
"""
from . import _lib, ops  # noqa: F401
from .model import ACR, Attention, Block, VisionTransformer  # noqa: F401
from .losses import acr_consistency_loss, acr_total_loss, dense_crf_loss, dense_crf_loss_from_patch_logits  # noqa: F401
from .cam import affinity_refine, infer_cam_image, infer_cam_batch, normalize_cam, pseudo_label, save_cam_dict, load_cam_dict, label_iou  # noqa: F401
from .cam import crf_inference, crf_with_alpha, crf_with_alpha_batch  # noqa: F401
from .pamr import PAMR  # noqa: F401
from .train import Trainer, PolyOptimizer  # noqa: F401
from .parallel import GradBuckets, shard_indices  # noqa: F401
from .bilateralfilter import bilateralfilter_batch, bilateralfilter  # noqa: F401
from .data import GpuAugment, Prefetcher, augment_params  # noqa: F401

__version__ = "0.1.0"
