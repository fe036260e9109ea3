"""sstem_restoration_b200 -- B200-native (sm_100a) hot path of ssTEM-restoration.

The package holds only what the path needs: the CUDA kernels and C ABI (csrc/,
include/sstem_b200.h), and the host-side mirrors of the reference's operator
interfaces:

    from sstem_restoration_b200 import SeparableConvolution          # libs/sepconv
    from sstem_restoration_b200 import FunctionSepconv, ModuleSepconv  # model/sepconv.py
    from sstem_restoration_b200 import SpatialTransformation, image_warp
    from sstem_restoration_b200 import interpolation_tail            # fused IFNet tail (model_interp.py:90-97)

There is no CPU / PyTorch fallback: without libsstem_b200.so (see
__graft_entry__.build) every operator raises.
"""
from ._lib import SstemError, launch_count, fp32_peak_probe  # noqa: F401
from .sepconv import (  # noqa: F401
    SeparableConvolution, FunctionSepconv, ModuleSepconv, set_strict_order, set_gray_replicated,
    interpolation_tail, ModuleInterpolationTail, taps_to_tiled, sepconv_forward_tiled,
    interpolation_tail_tiled, frame_mean_pad, taps_from_tiled, SeparableConvolutionTiled, ModuleInterpolationTailTiled,
)
from .warp import SpatialTransformation, image_warp  # noqa: F401
from .host import sepconv_forward_backward_host, join_host_pipeline  # noqa: F401
from .stack_io import sections_to_input, prediction_to_uint8  # noqa: F401
from .stack import restore_stack, warp_stitch, warp_and_stitch  # noqa: F401
from .tapconv import (  # noqa: F401
    tap_conv3x3, pack_tap_conv_weight, pack_tap_conv_weight_adjoint, TapConv3x3Function, ModuleTapProducer,
    branch_conv3x3, pack_branch_conv_weight, pack_branch_conv_weight_adjoint, branch_conv3x3_backward, ModuleTapBranch,
)
from . import shard, synth, sff_sim  # noqa: F401

__all__ = [
    "SeparableConvolution", "FunctionSepconv", "ModuleSepconv", "set_strict_order", "set_gray_replicated",
    "interpolation_tail", "ModuleInterpolationTail", "taps_to_tiled", "sepconv_forward_tiled", "interpolation_tail_tiled", "frame_mean_pad",
    "taps_from_tiled", "SeparableConvolutionTiled", "ModuleInterpolationTailTiled",
    "SpatialTransformation", "image_warp", "sepconv_forward_backward_host", "join_host_pipeline", "SstemError", "launch_count", "fp32_peak_probe",
    "sections_to_input", "prediction_to_uint8", "restore_stack", "warp_stitch", "warp_and_stitch",
    "tap_conv3x3", "pack_tap_conv_weight", "pack_tap_conv_weight_adjoint", "TapConv3x3Function", "ModuleTapProducer",
    "branch_conv3x3", "pack_branch_conv_weight", "pack_branch_conv_weight_adjoint", "branch_conv3x3_backward", "ModuleTapBranch", "shard", "synth", "sff_sim",
]
