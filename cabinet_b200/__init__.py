"""cabinet_b200 — B200-native forward hot path of CABiNet behind the reference's nn.Module surface."""

from .constants import BACKBONE_CFGS, DEFAULT_EVAL_SCALES, EVAL_STRIDE_RATE, MODEL_CONFIG  # noqa: F401
from .loss import OhemCELoss  # noqa: F401
from .modules import (AttentionBranch, CABiNet, CABiNetOutput, ContextAggregationBlock, FeatureFusionModule,  # noqa: F401
                      MobileNetV3, SpatialBranch)

__all__ = ["CABiNet", "ContextAggregationBlock", "MobileNetV3", "SpatialBranch", "AttentionBranch", "FeatureFusionModule",
           "CABiNetOutput", "OhemCELoss", "MODEL_CONFIG", "BACKBONE_CFGS", "EVAL_STRIDE_RATE", "DEFAULT_EVAL_SCALES"]
