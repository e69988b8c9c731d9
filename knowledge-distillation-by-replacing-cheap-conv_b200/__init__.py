"""kdcc -- B200-native (sm_100a) distillation hot path of "Knowledge Distillation by Replacing Cheap Conv".

Host-side mirror of the reference's module interfaces over the C-ABI library libkdcc.so
(include/kdcc.h).  The directory name carries the upstream repository name; import it as `kdcc`
(the top-level `kdcc/` shim registers this package under that name).
"""
from . import _abi
from ._abi import KdccError, LIB_PATH
from .blocks import DepthwiseSeparableBlock
from .losses import CrossEntropyLoss2d, EnsembleKLDivergenceLoss, KLDivergenceLoss, MSELoss, MultiTeacherKLDivergenceLoss, WeightedHintMSELoss
from . import checkpoint, functional, optim, tta
from .student import DepthwiseStudent
from .metrics import CityscapesMetricTracker, ConfusionMatrix
from .trainer import ClassificationStep, EnsembleStep, GradBucket, LayerwiseStep, prepare_train_epoch
from .peer_reduce import PeerGradBucket

__all__ = ["DepthwiseSeparableBlock", "DepthwiseStudent", "LayerwiseStep", "ClassificationStep", "EnsembleStep", "GradBucket", "PeerGradBucket", "prepare_train_epoch", "ConfusionMatrix", "CityscapesMetricTracker", "CrossEntropyLoss2d", "KLDivergenceLoss", "EnsembleKLDivergenceLoss", "MultiTeacherKLDivergenceLoss", "MSELoss", "WeightedHintMSELoss",
           "functional", "checkpoint", "KdccError", "LIB_PATH"]
