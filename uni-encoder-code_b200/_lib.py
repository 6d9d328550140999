"""ctypes loader for libmsda_b200.so (the C ABI declared in include/msda_b200.h).

There is deliberately no fallback: if the CUDA library is missing or fails to load,
importing this module raises, and every op in the package raises with it.
"""
from __future__ import annotations

import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
# MSDA_B200_LIB selects another build of the same ABI (the bounds-checked one of `make checked`)
LIB_PATH = os.environ.get("MSDA_B200_LIB") or os.path.join(_PKG, "lib", "libmsda_b200.so")

ABI_VERSION = 2

# name -> (restype, argtypes); must list every symbol of include/msda_b200.h
_P = ctypes.c_void_p
_I = ctypes.c_int
_DIMS = [_I] * 7
SYMBOLS = {
    "msda_b200_abi_version": (_I, []),
    "msda_b200_error_string": (ctypes.c_char_p, [_I]),
    "msda_b200_launch_count": (ctypes.c_longlong, []),
    "msda_b200_forward_f32": (_I, [_P] * 5 + _DIMS + [_P, _P]),
    "msda_b200_forward_f64": (_I, [_P] * 5 + _DIMS + [_P, _P]),
    "msda_b200_backward_f32": (_I, [_P] * 6 + _DIMS + [_P, _P, _P, _P]),
    "msda_b200_backward_f64": (_I, [_P] * 6 + _DIMS + [_P, _P, _P, _P]),
    "msda_b200_backward_deterministic_workspace_bytes": (ctypes.c_longlong, _DIMS + [_I]),
    "msda_b200_backward_deterministic_f32": (_I, [_P] * 6 + _DIMS + [_P, _P, _P, _P, _P]),
    "msda_b200_backward_deterministic_f64": (_I, [_P] * 6 + _DIMS + [_P, _P, _P, _P, _P]),
    "msda_b200_forward_bf16": (_I, [_P] * 5 + _DIMS + [_P, _P]),
    "msda_b200_forward_f16": (_I, [_P] * 5 + _DIMS + [_P, _P]),
    "msda_b200_backward_bf16": (_I, [_P] * 6 + _DIMS + [_P] * 5),
    "msda_b200_backward_f16": (_I, [_P] * 6 + _DIMS + [_P] * 5),
    "msda_b200_backward_deterministic_bf16": (_I, [_P] * 6 + _DIMS + [_P] * 5),
    "msda_b200_backward_deterministic_f16": (_I, [_P] * 6 + _DIMS + [_P] * 5),
    "msda_b200_debug_indices_f32": (_I, [_P] * 3 + _DIMS + [_P, _P, _P]),
    "msda_b200_fused_forward_f32": (_I, [_P] * 4 + [ctypes.c_longlong, _P, _P] + _DIMS + [_P, _P]),
    "msda_b200_fused_forward_strided_f32": (_I, [_P] * 4 + [ctypes.c_longlong, _P, _I, _P, _I, _P, _P] + _DIMS + [_P, _P]),
    "msda_b200_fused_backward_f32": (_I, [_P] * 5 + [ctypes.c_longlong, _P, _P] + _DIMS + [_P, _P, _P, _P]),
    "msda_b200_fused_backward_deterministic_f32": (_I, [_P] * 5 + [ctypes.c_longlong, _P, _P] + _DIMS + [_P] * 5),
    "msda_b200_fused_forward_bf16": (_I, [_P] * 4 + [ctypes.c_longlong, _P, _P] + _DIMS + [_P, _P]),
    "msda_b200_fused_forward_f16": (_I, [_P] * 4 + [ctypes.c_longlong, _P, _P] + _DIMS + [_P, _P]),
    "msda_b200_fused_backward_bf16": (_I, [_P] * 5 + [ctypes.c_longlong, _P, _P] + _DIMS + [_P] * 5),
    "msda_b200_fused_backward_f16": (_I, [_P] * 5 + [ctypes.c_longlong, _P, _P] + _DIMS + [_P] * 5),
    "msda_b200_fused_backward_deterministic_bf16": (_I, [_P] * 5 + [ctypes.c_longlong, _P, _P] + _DIMS + [_P] * 5),
    "msda_b200_fused_backward_deterministic_f16": (_I, [_P] * 5 + [ctypes.c_longlong, _P, _P] + _DIMS + [_P] * 5),
    "msda_b200_fused_forward_strided_bf16": (_I, [_P] * 4 + [ctypes.c_longlong, _P, _I, _P, _I, _P, _P] + _DIMS + [_P, _P]),
    "msda_b200_fused_forward_strided_f16": (_I, [_P] * 4 + [ctypes.c_longlong, _P, _I, _P, _I, _P, _P] + _DIMS + [_P, _P]),
    "msda_b200_linear_f32": (_I, [_P] * 4 + [_I] * 4 + [_P, _P]),
    "msda_b200_linear_deterministic_f32": (_I, [_P] * 4 + [_I] * 4 + [_P, _P]),
    "msda_b200_split_weight_f32": (_I, [_P, _P, _I, _I, _P]),
    "msda_b200_linear_presplit_f32": (_I, [_P] * 4 + [_I] * 4 + [_P]),
    "msda_b200_linear_presplit_deterministic_f32": (_I, [_P] * 4 + [_I] * 4 + [_P]),
    "msda_b200_add_layernorm_f32": (_I, [_P] * 5 + [ctypes.c_longlong, _I, ctypes.c_float, _P]),
    "msda_b200_add_layernorm_backward_f32": (_I, [_P] * 7 + [ctypes.c_longlong, _I, ctypes.c_float, _P]),
    "msda_b200_add_layernorm_backward_deterministic_f32": (_I, [_P] * 7 + [ctypes.c_longlong, _I, ctypes.c_float, _P, _P]),
    "msda_b200_add_layernorm_backward_deterministic_workspace_bytes": (ctypes.c_longlong, [ctypes.c_longlong, _I]),
    "msda_b200_add_layernorm_mixed_bf16": (_I, [_P] * 6 + [ctypes.c_longlong, _I, ctypes.c_float, _P]),
    "msda_b200_add_layernorm_mixed_f16": (_I, [_P] * 6 + [ctypes.c_longlong, _I, ctypes.c_float, _P]),
    "msda_b200_add_layernorm_mixed_backward_bf16": (_I, [_P] * 9 + [ctypes.c_longlong, _I, ctypes.c_float, _P]),
    "msda_b200_add_layernorm_mixed_backward_f16": (_I, [_P] * 9 + [ctypes.c_longlong, _I, ctypes.c_float, _P]),
    "msda_b200_add_layernorm_mixed_backward_deterministic_bf16": (_I, [_P] * 9 + [ctypes.c_longlong, _I, ctypes.c_float,
                                                                                 _P, _P]),
    "msda_b200_add_layernorm_mixed_backward_deterministic_f16": (_I, [_P] * 9 + [ctypes.c_longlong, _I, ctypes.c_float,
                                                                                _P, _P]),
    "msda_b200_linear_wgrad_f32": (_I, [_P] * 4 + [ctypes.c_longlong, _I, _I, _P]),
    "msda_b200_linear_wgrad_deterministic_f32": (_I, [_P] * 4 + [ctypes.c_longlong, _I, _I, _P, _P]),
    "msda_b200_linear_wgrad_deterministic_workspace_bytes": (ctypes.c_longlong, [ctypes.c_longlong, _I, _I]),
    "msda_b200_transpose_f32": (_I, [_P, _P, ctypes.c_longlong, _I, _P]),
    "msda_b200_linear_mixed_bf16": (_I, [_P] * 4 + [_I] * 4 + [_P]),
    "msda_b200_linear_mixed_f16": (_I, [_P] * 4 + [_I] * 4 + [_P]),
    "msda_b200_linear_mixed_wgrad_bf16": (_I, [_P] * 4 + [ctypes.c_longlong, _I, _I, _P, _P]),
    "msda_b200_linear_mixed_wgrad_f16": (_I, [_P] * 4 + [ctypes.c_longlong, _I, _I, _P, _P]),
    "msda_b200_linear_mixed_wgrad_workspace_bytes": (ctypes.c_longlong, [ctypes.c_longlong, _I, _I]),
    "msda_b200_group_norm_nchw_f32": (_I, [_P] * 5 + [_I] * 5 + [ctypes.c_float, _I, _P, _I, _I, _P, _P]),
    "msda_b200_group_norm_nchw_to_rows_f32": (_I, [_P] * 5 + [ctypes.c_longlong, ctypes.c_longlong, _I, _I, ctypes.c_longlong, _I,
                                                    ctypes.c_float, _I, _P, _P]),
    "msda_b200_add_channel_bias_nchw_f32": (_I, [_P, _P, _I, _I, ctypes.c_longlong, _P]),
    "msda_b200_group_norm_workspace_bytes": (ctypes.c_longlong, [_I, _I]),
    "msda_b200_group_norm_nchw_train_f32": (_I, [_P] * 6 + [_I] * 5 + [ctypes.c_float, _I, _P, _I, _I, _P, _P]),
    "msda_b200_group_norm_nchw_to_rows_train_f32": (_I, [_P] * 6 + [ctypes.c_longlong, ctypes.c_longlong, _I, _I,
                                                          ctypes.c_longlong, _I, ctypes.c_float, _I, _P, _P]),
    "msda_b200_group_norm_backward_nchw_f32": (_I, [_P] * 11 + [_I] * 8 + [_P, _P]),
    "msda_b200_group_norm_backward_workspace_bytes": (ctypes.c_longlong, [_I, _I]),
    "msda_b200_group_norm_rows_backward_f32": (_I, [_P, ctypes.c_longlong, ctypes.c_longlong] + [_P] * 9
                                               + [_I, _I, ctypes.c_longlong, _I, _I, _P, _P]),
    **{f"msda_b200_{name}_{sfx}": sig for sfx in ("bf16", "f16") for name, sig in (
        ("group_norm_nchw_mixed", (_I, [_P] * 6 + [_I] * 5 + [ctypes.c_float, _I, _P, _I, _I, _P, _P])),
        ("group_norm_nchw_mixed_train", (_I, [_P] * 7 + [_I] * 5 + [ctypes.c_float, _I, _P, _I, _I, _P, _P])),
        ("group_norm_nchw_to_rows_mixed", (_I, [_P] * 5 + [ctypes.c_longlong, ctypes.c_longlong, _I, _I,
                                                           ctypes.c_longlong, _I, ctypes.c_float, _I, _P, _P])),
        ("group_norm_nchw_to_rows_mixed_train", (_I, [_P] * 6 + [ctypes.c_longlong, ctypes.c_longlong, _I, _I,
                                                                 ctypes.c_longlong, _I, ctypes.c_float, _I, _P, _P])),
        ("group_norm_backward_nchw_mixed", (_I, [_P] * 12 + [_I] * 8 + [_P, _P])),
        ("group_norm_rows_backward_mixed", (_I, [_P, ctypes.c_longlong, ctypes.c_longlong] + [_P] * 9
                                            + [_I, _I, ctypes.c_longlong, _I, _I, _P, _P])),
        ("add_channel_bias_nchw", (_I, [_P, _P, _I, _I, ctypes.c_longlong, _P])))},
    "msda_b200_set_option": (_I, [ctypes.c_char_p, _I]),
    "msda_b200_get_option": (_I, [ctypes.c_char_p, ctypes.POINTER(_I)]),
}


class MSDALibraryError(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into lib/libmsda_b200.so (nvcc, no GPU needed)."""
    import subprocess
    res = subprocess.run(["make", "-C", os.path.join(_PKG, "csrc"), "-j4"],
                         capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout + res.stderr)
    if res.returncode != 0:
        raise MSDALibraryError("building libmsda_b200.so failed (see output above)")
    return LIB_PATH


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise MSDALibraryError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C uni-encoder-code_b200/csrc`. There is no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    got = lib.msda_b200_abi_version()
    if got != ABI_VERSION:
        raise MSDALibraryError(f"libmsda_b200.so ABI {got} != expected {ABI_VERSION}; rebuild")
    return lib


lib = _load()


def check(code: int, what: str) -> None:
    if code != 0:
        msg = lib.msda_b200_error_string(code).decode()
        raise RuntimeError(f"{what} failed: {msg} (code {code})")


def set_option(name: str, value: int) -> None:
    check(lib.msda_b200_set_option(name.encode(), int(value)), f"set_option({name})")


def get_option(name: str) -> int:
    v = _I(0)
    check(lib.msda_b200_get_option(name.encode(), ctypes.byref(v)), f"get_option({name})")
    return v.value


def launch_count() -> int:
    return int(lib.msda_b200_launch_count())
