"""rdvc_corr_b200 -- B200-native RAFT correlation hot path for RDVC's motion branch.

The directory is named after the reference repository
(``pfe-raft-and-hyperprior-based-learned-video-compression_b200``), which is not a
valid Python identifier; import it through the root-level shim::

    import rdvc_corr_b200 as rc
    blk = rc.TVCorrBlock()                       # torchvision surface
    corr = rc.CorrBlock(fmap1, fmap2, 4, 4)      # princeton-style façade
    feats = corr(coords)

Contents: ``csrc/`` (hand-written sm_100a kernels + the C ABI of
``include/rdvc_corr.h``), ``_build`` (nvcc driver), ``_cabi`` (ctypes binding),
``corr_block`` (host-side mirror of the reference interface).
"""
from . import _build, _cabi, entropy_coder, gop_shard, rdvc_format  # noqa: F401
from ._cabi import (RDVC_DT_BF16, RDVC_DT_F16, RDVC_DT_F32,  # noqa: F401
                    RDVC_LAYOUT_ROWMAJOR, RDVC_LAYOUT_TILED)
from .corr_block import (  # noqa: F401
    CorrBlock,
    CorrPyramid,
    TVCorrBlock,
    build_pyramid,
    index_pyramid,
)
from .context_encoder import ContextEncoder  # noqa: F401
from .feature_encoder import FeatureEncoder  # noqa: F401
from .mask_predictor import MaskPredictor  # noqa: F401
from .mcn import MotionCompensationNetwork  # noqa: F401
from .motion_encoder import FlowHead, MotionEncoder  # noqa: F401
from .motion_warp import WarpingLayer, motion_warp, resize_flow  # noqa: F401
from .preprocess import frame_to_tensor, preprocess_frame_codec, preprocess_frame_raft  # noqa: F401
from .raft_flow import GraphedRaftFlow, raft_flow, raft_flow_sequence  # noqa: F401
from .recurrent_block import RecurrentBlock  # noqa: F401

__all__ = [
    "CorrBlock", "CorrPyramid", "TVCorrBlock", "build_pyramid", "index_pyramid", "raft_flow", "raft_flow_sequence", "GraphedRaftFlow",
    "WarpingLayer", "motion_warp", "resize_flow", "MotionCompensationNetwork", "RecurrentBlock",
    "MotionEncoder", "FlowHead", "MaskPredictor", "ContextEncoder", "FeatureEncoder",
    "frame_to_tensor", "preprocess_frame_codec", "preprocess_frame_raft",
    "RDVC_DT_BF16", "RDVC_DT_F16", "RDVC_DT_F32", "RDVC_LAYOUT_ROWMAJOR", "RDVC_LAYOUT_TILED",
]
