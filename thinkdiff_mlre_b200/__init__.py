"""thinkdiff_mlre_b200 -- B200-native (sm_100a) implementation of the ThinkDiff aligner hot path.

pack (ragged, cu_seqlens) -> Linear -> GELU -> Linear -> T5 RMSNorm (forward / backward on tcgen05 + TMA) -> masked
MSE / cross-entropy -> data-parallel gradient all-reduce, behind the reference's ``mm_projector`` nn.Module boundary.
Importing the package loads ``libthinkdiff_b200.so``; if it is not built the import fails -- there is no fallback.
"""
from . import _lib

_lib.lib()  # fail loudly at import time when the CUDA library is missing

from . import ops  # noqa: E402
from .aligner import FUSED_TYPE, ThinkDiffAligner, build_vision_projector  # noqa: E402
from .loss import frozen_linear, lm_head_cross_entropy, masked_cross_entropy, masked_mse  # noqa: E402
from .pack import FlatBatch, FlatCollater, PackedBatch, compose_image_text, kept_lengths, pack_batch, pack_device  # noqa: E402
from .train_step import AlignerTrainStep, synthetic_lvlm_batch  # noqa: E402
from .optim import DeviceGradScaler, FusedAdamW  # noqa: E402
from .shards import EmbedShardReader, EmbedShardSet, EmbedShardWriter, convert_webdataset_shards, iter_webdataset_samples  # noqa: E402
from .lr_schedule import LinearWarmupCosineLRScheduler, LinearWarmupStepLRScheduler, get_lr_scheduler_class  # noqa: E402
from .t5 import T5FeedForwardWeights, t5_attention, t5_layer_ff, t5_position_bias_by_distance  # noqa: E402

__all__ = [
    "ops", "ThinkDiffAligner", "build_vision_projector", "FUSED_TYPE", "masked_mse", "masked_cross_entropy", "lm_head_cross_entropy", "frozen_linear",
    "FlatBatch", "FlatCollater", "PackedBatch", "kept_lengths", "pack_batch", "pack_device", "compose_image_text", "AlignerTrainStep",
    "synthetic_lvlm_batch", "FusedAdamW", "DeviceGradScaler", "EmbedShardReader", "EmbedShardSet", "EmbedShardWriter", "convert_webdataset_shards", "iter_webdataset_samples", "LinearWarmupCosineLRScheduler",
    "LinearWarmupStepLRScheduler", "get_lr_scheduler_class", "t5_attention", "t5_position_bias_by_distance", "t5_layer_ff",
    "T5FeedForwardWeights",
]
