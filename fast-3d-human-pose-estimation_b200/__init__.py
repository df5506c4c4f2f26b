"""B200-native CDRNet post-backbone hot path (sm_100a) behind the reference's Python interfaces.

    from fast_3d_human_pose_estimation_b200 import CDRNet, PoseResNet, calc_mpjpe, \
        get_max_preds, triangulation

mirrors ``models.cdrnet.CDRNet``, ``models.poseresnet.PoseResNet``, ``models.metrics.calc_mpjpe``,
``tools.utils.get_max_preds`` and ``tools.common.triangulation`` of
eddie0509tw/Fast-3D-Human-Pose-Estimation (see INTEGRATION.md).  All arithmetic after the ResNet
encoder runs in libcdrhead.so (include/cdrhead.h); there is no CPU or PyTorch fallback.
"""
from . import _lib
from ._lib import CdrError, build
from .cdrnet import CDRNet, CanonicalFusion, PoseDecoder, PoseResNet
from .encoder import ResNet
from .graph import HeadGraph, HeadPipeline, FramePipeline
from .geometry import baseline_keypoints, get_max_preds, projection_matrices, triangulation
from .metrics import calc_mpjpe, mpjpe_sums
from .autograd import soft_argmax_2d, dlt, ftl, conv_transpose2d, conv1x1, conv3x3, stem_conv, max_pool3x3
from .losses import JointsMSELoss, JointsMSESmoothLoss, MPJPELoss, batch_norm_train

__all__ = ["CDRNet", "CanonicalFusion", "PoseDecoder", "PoseResNet", "ResNet", "calc_mpjpe",
           "mpjpe_sums", "HeadGraph", "HeadPipeline", "FramePipeline", "get_max_preds", "baseline_keypoints", "triangulation", "soft_argmax_2d", "dlt", "ftl", "conv_transpose2d", "conv1x1", "conv3x3", "stem_conv", "max_pool3x3", "JointsMSELoss", "JointsMSESmoothLoss", "MPJPELoss", "batch_norm_train", "build",
           "CdrError"]
