"""B200-native multi-scale deformable attention -- drop-in for the MSDeformAttn hot path of
yunduo-vision/IR-ADS (detrex.layers.MultiScaleDeformableAttention and the
ms_deform_attn_forward / backward CUDA pair) -- plus DCNv3 and detectron2's deformable convolution
(DeformConv / ModulatedDeformConv).  See DESIGN.md and include/msda.h.

Importing the package does not load the CUDA library; the first op call does, and fails loudly
if ir_ads_b200/libmsda_b200.so has not been built (no CPU / PyTorch fallback exists).
"""
from .functional import (  # noqa: F401
    MSDeformAttnPackedFunction,
    MultiScaleDeformableAttnFunction,
    kernel_flags,
    ms_deform_attn_backward,
    ms_deform_attn_forward,
    multi_scale_deformable_attn_pytorch,
    set_deterministic,
)
from .dcnv2 import DCNv2Function, DeformConv, ModulatedDeformConv, deform_conv, modulated_deform_conv  # noqa: F401
from .dcnv3 import DCNv3FusedFunction, DCNv3Function, dcnv3_backward, dcnv3_forward  # noqa: F401
from .module import MultiScaleDeformableAttention  # noqa: F401
from .packing import PackedLevels, pack_levels, packed_reference_points, unpack_tokens, valid_extents  # noqa: F401
from . import ops  # noqa: F401,E402  (registers the torch.library custom ops; loads no library)

__all__ = [
    "MultiScaleDeformableAttention",
    "MultiScaleDeformableAttnFunction",
    "ms_deform_attn_forward",
    "ms_deform_attn_backward",
    "multi_scale_deformable_attn_pytorch",
    "set_deterministic",
    "kernel_flags",
    "DeformConv",
    "ModulatedDeformConv",
    "deform_conv",
    "modulated_deform_conv",
    "DCNv2Function",
    "DCNv3Function",
    "DCNv3FusedFunction",
    "dcnv3_forward",
    "dcnv3_backward",
    "MSDeformAttnPackedFunction",
    "PackedLevels",
    "valid_extents",
    "pack_levels",
    "packed_reference_points",
    "unpack_tokens",
    "ops",
]
