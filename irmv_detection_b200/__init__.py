"""irmv_detection_b200 -- B200-native (sm_100a) per-frame armor pipeline behind the reference's
YoloEngine / PnPSolver interfaces.  All compute is in libirmv_b200.so (hand-written CUDA); see
DESIGN.md and include/irmv_cabi.h."""
from ._lib import (CH_BAYER_BGGR, CH_BAYER_GBRG, CH_BAYER_GRBG, CH_BAYER_RGGB, CH_PASSTHROUGH,
                   CH_SWAP_RB, CONV_DIRECT, CONV_TCGEN05, RAW_8, RAW_10, RAW_12, RAW_12_PACKED, IrmvError)
from .engine import (ARMOR_DTYPE, AWB_DTYPE, BBOX_DTYPE, POSE_DTYPE, ArmorClass, PnPSolver, YoloEngine, armor_params, bbox, decode,
                     extract_armors, nms, preprocess)

__all__ = ["YoloEngine", "PnPSolver", "ArmorClass", "bbox", "preprocess", "nms", "decode", "extract_armors", "armor_params", "ARMOR_DTYPE", "AWB_DTYPE", "BBOX_DTYPE", "POSE_DTYPE", "IrmvError",
           "CH_PASSTHROUGH", "CH_SWAP_RB", "CH_BAYER_RGGB", "CH_BAYER_BGGR", "CH_BAYER_GRBG",
           "CH_BAYER_GBRG", "CONV_TCGEN05", "CONV_DIRECT", "RAW_8", "RAW_10", "RAW_12", "RAW_12_PACKED"]
