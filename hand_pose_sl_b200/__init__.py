"""hand_pose_sl_b200 -- B200 (sm_100a) native hot path of benoriol/hand_pose_sl's body2hand:
temporal-conv regressor, masked-L1 train step and keypoint preprocessing behind the reference's own
nn.Module / criterion / transform API.  All compute is in libb2h.so (hand-written CUDA, C-ABI in
include/b2h.h); there is no CPU fallback."""
from . import _lib, synthetic  # noqa: F401
from .models import ConvModel, LinearPositionalEmbedding, format_prediction  # noqa: F401
from .steps import (FusedAdam, L12Pixels, adjust_learning_rate, forward_backward, forward_backward_utterances,  # noqa: F401
                    forward_backward_windows, fused_train_step, fused_train_step_utterances, fused_train_step_windows,
                    mask_output, maskedPoseL1, poderatedPoseL1, validate_batch, validate_utterances)
from .datasets import GpuPoseDataset, PackedClips, pack_metadata, split_metadata  # noqa: F401
from .transforms import BODY_HEAD_KEYPOINTS, PreprocessRightHand, select_window, sliding_window_starts  # noqa: F401

fused_step = fused_train_step      # the name SURVEY.md 8b uses for the optional one-call fast path

__all__ = ["fused_step", "ConvModel", "LinearPositionalEmbedding", "maskedPoseL1", "poderatedPoseL1", "mask_output", "FusedAdam",
           "fused_train_step", "forward_backward", "fused_train_step_windows", "forward_backward_windows",
           "fused_train_step_utterances", "forward_backward_utterances", "validate_batch",
           "validate_utterances", "PreprocessRightHand", "select_window",
           "sliding_window_starts", "L12Pixels", "adjust_learning_rate", "BODY_HEAD_KEYPOINTS", "GpuPoseDataset", "PackedClips",
           "pack_metadata", "split_metadata", "format_prediction"]
