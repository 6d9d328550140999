"""msda-b200: B200-native (sm_100a) multi-scale deformable attention behind the
reference's ``MultiScaleDeformableAttention`` plugin API.

Importing this package loads ``lib/libmsda_b200.so`` through ctypes and raises if it
is missing -- there is no CPU or PyTorch fallback anywhere in the package.

Public surface (names mirror the reference, see INTEGRATION.md):
    ms_deform_attn_forward / ms_deform_attn_backward   (ops/src/vision.cpp:18-21)
    MSDeformAttnFunction                               (ops/functions/ms_deform_attn_func.py:35-52)
    MSDeformAttnMixedFunction -- the same op for bf16 / fp16 value rows (torch.autocast)
    install_dropin()  -- makes ``import MultiScaleDeformableAttention`` resolve to the shim
"""
from __future__ import annotations

import os
import sys

from . import _lib
from ._lib import get_option, launch_count, set_option
from .functions import (AddLayerNormFunction, AddLayerNormMixedFunction, GroupNormFunction, GroupNormRowsFunction, LinearMixedFunction,
                        LinearTF32x3Function, MSDeformAttnFunction, MSDeformAttnFusedFunction, MSDeformAttnMixedFunction)
from .ops import (add_layernorm, add_layernorm_mixed, debug_indices, group_norm, linear_mixed, linear_tf32x3, ms_deform_attn_backward, ms_deform_attn_forward,
                  ms_deform_attn_fused_backward, ms_deform_attn_fused_forward, ms_deform_attn_mixed_backward,
                  ms_deform_attn_mixed_forward)
from . import synthetic
from . import modules, pixel_decoder, sharding

__all__ = [
    "ms_deform_attn_forward", "ms_deform_attn_backward", "MSDeformAttnFunction", "debug_indices",
    "ms_deform_attn_fused_forward", "ms_deform_attn_fused_backward", "MSDeformAttnFusedFunction", "linear_tf32x3", "add_layernorm", "group_norm", "LinearTF32x3Function", "AddLayerNormFunction",
    "GroupNormFunction", "GroupNormRowsFunction",
    "ms_deform_attn_mixed_forward", "ms_deform_attn_mixed_backward", "MSDeformAttnMixedFunction",
    "add_layernorm_mixed", "AddLayerNormMixedFunction", "linear_mixed", "LinearMixedFunction",
    "install_dropin", "set_option", "get_option", "launch_count", "synthetic", "modules", "pixel_decoder", "sharding",
]

DROPIN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "dropin")


def install_dropin() -> str:
    """Put the ``MultiScaleDeformableAttention`` shim first on sys.path (idempotent).

    Call before importing the reference's ``ops.functions`` (func.py:21-30 imports the
    module at import time when CUDA is available)."""
    if DROPIN_DIR not in sys.path:
        sys.path.insert(0, DROPIN_DIR)
    return DROPIN_DIR
