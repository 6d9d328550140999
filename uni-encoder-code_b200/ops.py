"""Host side of the drop-in boundary: the two functions the reference's pybind11 module
``MultiScaleDeformableAttention`` exports (ops/src/vision.cpp:18-21), re-implemented as
thin Python over the C ABI (include/msda_b200.h).

Argument meaning, order, return types and error behaviour follow the reference's
dispatch + host wrappers (ops/src/ms_deform_attn.h:25-66,
ops/src/cuda/ms_deform_attn_cuda.cu:25-85 and :88-158):

* a non-CUDA ``value`` raises ``RuntimeError("Not implemented on the CPU")``
  (ms_deform_attn.h:43,65) -- there is no CPU path here either;
* every tensor must be contiguous and on a CUDA device (cu:33-43, :98-110);
* ``im2col_step_ = min(batch, im2col_step)`` must divide ``batch`` (cu:55-57, :122-124).
  It is validated for error parity and otherwise ignored: one launch covers the batch;
* dtype float32 or float64 (AT_DISPATCH_FLOATING_TYPES, cu:69,139); the shape tensors
  are int64 on the device (``.data<int64_t>()``, cu:72-73);
* outputs are allocated here with torch's caching allocator on the current stream
  (the reference allocates with ``value.options()``, cu:59, :126-128); the C side never
  allocates, frees or synchronises.
"""
from __future__ import annotations

import torch

from . import _lib

# Optional per-call CUDA-event timing of the two C-ABI launches (bench tools only; off by
# default, no effect on results).  When enabled, every call appends (kind, start, end).
_TIMING = None


def enable_timing(on: bool = True):
    """Start (or stop) collecting CUDA events around each kernel launch; returns the list."""
    global _TIMING
    _TIMING = [] if on else None
    return _TIMING


class _timed:
    def __init__(self, kind):
        self.kind = kind

    def __enter__(self):
        if _TIMING is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()

    def __exit__(self, *exc):
        if _TIMING is not None:
            self.e1.record()
            _TIMING.append((self.kind, self.e0, self.e1))


_FWD = {torch.float32: _lib.lib.msda_b200_forward_f32, torch.float64: _lib.lib.msda_b200_forward_f64}
_BWD = {torch.float32: _lib.lib.msda_b200_backward_f32, torch.float64: _lib.lib.msda_b200_backward_f64}
_BWD_DET = {torch.float32: _lib.lib.msda_b200_backward_deterministic_f32,
            torch.float64: _lib.lib.msda_b200_backward_deterministic_f64}
# the mixed-precision op: 16-bit value / output / grad_output / grad_value, fp32 locations and weights
_MIXED_FWD = {torch.bfloat16: _lib.lib.msda_b200_forward_bf16, torch.float16: _lib.lib.msda_b200_forward_f16}
_MIXED_BWD = {torch.bfloat16: _lib.lib.msda_b200_backward_bf16, torch.float16: _lib.lib.msda_b200_backward_f16}
_MIXED_BWD_DET = {torch.bfloat16: _lib.lib.msda_b200_backward_deterministic_bf16,
                  torch.float16: _lib.lib.msda_b200_backward_deterministic_f16}

# With torch.use_deterministic_algorithms(True) every backward here takes its deterministic entry point.  The
# MSDA backwards then sort one record per (sampling point, corner): the batch is processed in chunks of whole
# images of at most this many records (20 bytes each in fp32, plus the sort's scratch), which bounds the
# workspace and keeps the record slots 32-bit.  Chunks write disjoint grad_value rows, so the chunking cannot
# change a bit of the result.
DETERMINISTIC_RECORD_LIMIT = 1 << 25


def _deterministic() -> bool:
    return torch.are_deterministic_algorithms_enabled()


def _image_chunks(N, records_per_image):
    step = max(1, min(N, DETERMINISTIC_RECORD_LIMIT // records_per_image))
    return [(n0, min(N, n0 + step)) for n0 in range(0, N, step)]


def _det_workspace(images, S, M, D, L, Lq, P, dtype, device):
    nbytes = _lib.lib.msda_b200_backward_deterministic_workspace_bytes(images, S, M, D, L, Lq, P,
                                                                       torch.empty((), dtype=dtype).element_size())
    if nbytes <= 0:
        raise RuntimeError("deterministic MSDA backward: one image has more than 2^31 - 1 corner records")
    return torch.empty(int(nbytes), dtype=torch.uint8, device=device)


def _require_cuda_contiguous(named):
    """The reference's input checks over (name, tensor) pairs: every tensor contiguous and on the device of the
    first one, which must be a CUDA tensor."""
    first, anchor = named[0]
    if not isinstance(anchor, torch.Tensor) or not anchor.is_cuda:
        raise RuntimeError("Not implemented on the CPU")                     # ms_deform_attn.h:43,65
    for name, t in named:
        if not t.is_contiguous():
            raise RuntimeError(f"{name} tensor has to be contiguous")        # cu:33-37
    for name, t in named:
        if not t.is_cuda:
            raise RuntimeError(f"{name} must be a CUDA tensor")              # cu:39-43
        if t.device != anchor.device:
            raise RuntimeError(f"{name} is on {t.device}, {first} is on {anchor.device}")


def _check_common(named, im2col_step, opname, mixed=False):
    """The checks of the op over (name, tensor) pairs (value, spatial_shapes, level_start_index, sampling_loc,
    attn_weight[, grad_output]) -> (N, S, M, D, L, Lq, P).  ``mixed``: the mixed-precision op's dtypes -- a 16-bit
    value (and grad_output of the same type), fp32 sampling_loc and attn_weight."""
    _require_cuda_contiguous(named)
    value = named[0][1]
    if value.dtype not in (_MIXED_FWD if mixed else _FWD):
        raise RuntimeError(f'"{opname}" not implemented for \'{value.dtype}\'')   # cu:69,139
    _, shapes, lsi, loc, w = (t for _, t in named[:5])
    for name, t in named[1:3]:
        if t.dtype != torch.int64:
            raise RuntimeError(f"expected scalar type Long but found {t.dtype} for {name}")
    for i, (name, t) in enumerate(named[3:], start=3):
        want = torch.float32 if mixed and i < 5 else value.dtype
        if t.dtype != want:
            hint = " (the mixed-precision op keeps locations and weights in fp32)" if want == torch.float32 and mixed else ""
            raise RuntimeError(f"expected scalar type {want} but found {t.dtype} for {name}{hint}")
    if value.dim() != 4 or loc.dim() != 6 or shapes.dim() != 2 or shapes.size(1) != 2:
        raise RuntimeError("value must be [N,S,M,D], sampling_loc [N,Lq,M,L,P,2], spatial_shapes [L,2]")
    N, S, M, D = value.shape
    L = shapes.size(0)
    Lq, P = loc.size(1), loc.size(4)
    if tuple(loc.shape) != (N, Lq, M, L, P, 2) or w.numel() != N * Lq * M * L * P or lsi.numel() != L:
        raise RuntimeError(
            f"inconsistent shapes: value {tuple(value.shape)}, spatial_shapes {tuple(shapes.shape)}, "
            f"level_start_index {tuple(lsi.shape)}, sampling_loc {tuple(loc.shape)}, "
            f"attn_weight {tuple(w.shape)}")
    step = min(N, int(im2col_step))
    if N == 0:
        return N, S, M, D, L, Lq, P
    if step <= 0 or N % step != 0:
        raise RuntimeError(f"batch({N}) must divide im2col_step({step})")     # cu:57, :124
    return N, S, M, D, L, Lq, P


def ms_deform_attn_forward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight,
                           im2col_step):
    """-> output [N, Lq, M*D]  (vision.cpp:19; ms_deform_attn_cuda.cu:25-85)."""
    named = [("value", value), ("spatial_shapes", spatial_shapes),
             ("level_start_index", level_start_index), ("sampling_loc", sampling_loc),
             ("attn_weight", attn_weight)]
    N, S, M, D, L, Lq, P = _check_common(named, im2col_step, "ms_deform_attn_forward_cuda")
    if N * Lq * M * D == 0 or S == 0 or L * P == 0:
        # nothing to sample: the reference returns its zero-initialised output (cu:59)
        return torch.zeros((N, Lq, M * D), dtype=value.dtype, device=value.device)
    with torch.cuda.device(value.device):
        output = torch.empty((N, Lq, M * D), dtype=value.dtype, device=value.device)
        with _timed("forward"):
            rc = _FWD[value.dtype](
                value.data_ptr(), spatial_shapes.data_ptr(), level_start_index.data_ptr(),
                sampling_loc.data_ptr(), attn_weight.data_ptr(), N, S, M, D, L, Lq, P,
                output.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "ms_deform_attn_forward")
    return output


def ms_deform_attn_backward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight,
                            grad_output, im2col_step):
    """-> [grad_value, grad_sampling_loc, grad_attn_weight]  (vision.cpp:20; cu:88-158)."""
    named = [("value", value), ("spatial_shapes", spatial_shapes),
             ("level_start_index", level_start_index), ("sampling_loc", sampling_loc),
             ("attn_weight", attn_weight), ("grad_output", grad_output)]
    N, S, M, D, L, Lq, P = _check_common(named, im2col_step, "ms_deform_attn_backward_cuda")
    if grad_output.numel() != N * Lq * M * D:
        raise RuntimeError(f"grad_output has {grad_output.numel()} elements, expected {N * Lq * M * D}")
    if N * Lq * M * D == 0 or S == 0 or L * P == 0:
        # nothing to sample: all three gradients stay at the reference's zero fill (cu:126-128)
        return [torch.zeros_like(value), torch.zeros_like(sampling_loc), torch.zeros_like(attn_weight)]
    if _deterministic():
        return _backward_deterministic(_BWD_DET[value.dtype], "ms_deform_attn_backward (deterministic)", value,
                                       spatial_shapes, level_start_index, (sampling_loc, attn_weight), grad_output,
                                       (N, S, M, D, L, Lq, P))
    with torch.cuda.device(value.device):
        grad_value = torch.zeros_like(value)            # accumulated by reductions (cu:126)
        grad_loc = torch.empty_like(sampling_loc)       # fully overwritten (cf. cu:127)
        grad_w = torch.empty_like(attn_weight)          # fully overwritten (cf. cu:128)
        with _timed("backward"):
            rc = _BWD[value.dtype](
                grad_output.data_ptr(), value.data_ptr(), spatial_shapes.data_ptr(),
                level_start_index.data_ptr(), sampling_loc.data_ptr(), attn_weight.data_ptr(),
                N, S, M, D, L, Lq, P, grad_value.data_ptr(), grad_loc.data_ptr(), grad_w.data_ptr(),
                torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "ms_deform_attn_backward")
    return [grad_value, grad_loc, grad_w]


def _backward_deterministic(fn, opname, value, shapes, lsi, producers, grad_output, dims, ref=None, rs=0,
                            kind="backward"):
    """A deterministic backward entry ``fn`` (msda_b200_backward_deterministic_f32/_f64/_bf16/_f16, or with ``ref`` the fused
    msda_b200_fused_backward_deterministic_f32/_bf16/_f16) in chunks of whole images -> [grad_value, *grads of producers].
    ``producers``: (sampling_loc, attn_weight), or for the fused op (sampling_offsets, attn_logits).  ``kind``: the
    name of the call in ``enable_timing``'s list, the same as the default backward's."""
    N, S, M, D, L, Lq, P = dims
    chunks = _image_chunks(N, Lq * M * L * P * 4)
    with torch.cuda.device(value.device):
        grad_value = torch.empty_like(value)            # fully overwritten by the gather
        grads = [torch.empty_like(t) for t in producers]
        ws = _det_workspace(max(b - a for a, b in chunks), S, M, D, L, Lq, P, value.dtype, value.device)
        stream = torch.cuda.current_stream().cuda_stream
        with _timed(kind):
            for a, b in chunks:
                fused = ()
                if ref is not None:                     # rs == 0: one set of reference points shared by the batch
                    fused = ((ref[a:b] if rs != 0 and ref.size(0) == N else ref).data_ptr(), rs)
                rc = fn(grad_output[a:b].data_ptr(), value[a:b].data_ptr(), shapes.data_ptr(), lsi.data_ptr(), *fused,
                        *(t[a:b].data_ptr() for t in producers), b - a, S, M, D, L, Lq, P, grad_value[a:b].data_ptr(),
                        *(g[a:b].data_ptr() for g in grads), ws.data_ptr(), stream)
                _lib.check(rc, opname)
    return [grad_value, *grads]


# ----------------------------------------------------------------------------------------------
# Mixed precision (torch.autocast): bf16 / fp16 value rows with fp32 locations, weights and sums.  Not part of the
# drop-in boundary above, which keeps the reference's fp32 / fp64 dtype contract.
# ----------------------------------------------------------------------------------------------
def ms_deform_attn_mixed_forward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, im2col_step):
    """-> output [N, Lq, M*D] in value's dtype, for a bf16 / fp16 ``value`` and fp32 ``sampling_loc`` /
    ``attn_weight``: the fp32 op on the widened value, rounded once to the 16-bit type (msda_b200_forward_bf16 /
    _f16).  Arguments as ``ms_deform_attn_forward``; ``im2col_step`` is validated and ignored."""
    named = [("value", value), ("spatial_shapes", spatial_shapes),
             ("level_start_index", level_start_index), ("sampling_loc", sampling_loc),
             ("attn_weight", attn_weight)]
    N, S, M, D, L, Lq, P = _check_common(named, im2col_step, "ms_deform_attn_mixed_forward", mixed=True)
    if N * Lq * M * D == 0 or S == 0 or L * P == 0:
        return torch.zeros((N, Lq, M * D), dtype=value.dtype, device=value.device)
    with torch.cuda.device(value.device):
        output = torch.empty((N, Lq, M * D), dtype=value.dtype, device=value.device)
        with _timed("forward_mixed"):
            rc = _MIXED_FWD[value.dtype](
                value.data_ptr(), spatial_shapes.data_ptr(), level_start_index.data_ptr(),
                sampling_loc.data_ptr(), attn_weight.data_ptr(), N, S, M, D, L, Lq, P,
                output.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "ms_deform_attn_mixed_forward")
    return output


def ms_deform_attn_mixed_backward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight,
                                  grad_output, im2col_step):
    """-> [grad_value (value's dtype), grad_sampling_loc, grad_attn_weight (fp32)] of the mixed-precision op.
    grad_value is reduced in an fp32 buffer allocated here and rounded once (msda_b200_backward_bf16 / _f16); with
    torch.use_deterministic_algorithms(True) the deterministic entries, in image chunks as for fp32."""
    named = [("value", value), ("spatial_shapes", spatial_shapes),
             ("level_start_index", level_start_index), ("sampling_loc", sampling_loc),
             ("attn_weight", attn_weight), ("grad_output", grad_output)]
    N, S, M, D, L, Lq, P = _check_common(named, im2col_step, "ms_deform_attn_mixed_backward", mixed=True)
    if grad_output.numel() != N * Lq * M * D:
        raise RuntimeError(f"grad_output has {grad_output.numel()} elements, expected {N * Lq * M * D}")
    if N * Lq * M * D == 0 or S == 0 or L * P == 0:
        return [torch.zeros_like(value), torch.zeros_like(sampling_loc), torch.zeros_like(attn_weight)]
    if _deterministic():
        return _backward_deterministic(_MIXED_BWD_DET[value.dtype], "ms_deform_attn_mixed_backward (deterministic)",
                                       value, spatial_shapes, level_start_index, (sampling_loc, attn_weight),
                                       grad_output, (N, S, M, D, L, Lq, P), kind="backward_mixed")
    with torch.cuda.device(value.device):
        accum = torch.zeros((N, S, M, D), dtype=torch.float32, device=value.device)   # fp32 reductions
        grad_value = torch.empty_like(value)            # rounded from accum
        grad_loc = torch.empty_like(sampling_loc)
        grad_w = torch.empty_like(attn_weight)
        with _timed("backward_mixed"):
            rc = _MIXED_BWD[value.dtype](
                grad_output.data_ptr(), value.data_ptr(), spatial_shapes.data_ptr(),
                level_start_index.data_ptr(), sampling_loc.data_ptr(), attn_weight.data_ptr(),
                N, S, M, D, L, Lq, P, accum.data_ptr(), grad_value.data_ptr(), grad_loc.data_ptr(),
                grad_w.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "ms_deform_attn_mixed_backward")
    return [grad_value, grad_loc, grad_w]


def debug_indices(value_shape, spatial_shapes, level_start_index, sampling_loc):
    """Integer known-answer hook (msda_b200_debug_indices_f32): (idx int32 [...,4], off int64 [...,4])."""
    N, S, M, D = (int(x) for x in value_shape)
    if not sampling_loc.is_cuda or sampling_loc.dtype != torch.float32 or not sampling_loc.is_contiguous():
        raise RuntimeError("sampling_loc must be a contiguous float32 CUDA tensor")
    L = spatial_shapes.size(0)
    Lq, P = sampling_loc.size(1), sampling_loc.size(4)
    with torch.cuda.device(sampling_loc.device):
        idx = torch.empty(tuple(sampling_loc.shape[:-1]) + (4,), dtype=torch.int32, device=sampling_loc.device)
        off = torch.empty(tuple(sampling_loc.shape[:-1]) + (4,), dtype=torch.int64, device=sampling_loc.device)
        rc = _lib.lib.msda_b200_debug_indices_f32(
            spatial_shapes.data_ptr(), level_start_index.data_ptr(), sampling_loc.data_ptr(),
            N, S, M, D, L, Lq, P, idx.data_ptr(), off.data_ptr(),
            torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "debug_indices")
    return idx, off


# ----------------------------------------------------------------------------------------------
# Fused producers (SURVEY.md 8f.1): softmax over the L*P logits and `ref + offset / (W, H)` inside
# the kernels (ops/modules/ms_deform_attn.py:105-112).  No counterpart in the reference's extension.
# ----------------------------------------------------------------------------------------------
# the mixed-precision fused op (torch.autocast): 16-bit value, raw offsets / logits and their gradients, fp32 reference
# points, fp32 arithmetic in between
_FUSED_MIXED_FWD = {torch.bfloat16: _lib.lib.msda_b200_fused_forward_bf16,
                    torch.float16: _lib.lib.msda_b200_fused_forward_f16}
_FUSED_MIXED_BWD = {torch.bfloat16: _lib.lib.msda_b200_fused_backward_bf16,
                    torch.float16: _lib.lib.msda_b200_fused_backward_f16}
_FUSED_MIXED_BWD_DET = {torch.bfloat16: _lib.lib.msda_b200_fused_backward_deterministic_bf16,
                        torch.float16: _lib.lib.msda_b200_fused_backward_deterministic_f16}


def fused_supported(value, reference_points, sampling_offsets, attn_logits):
    """The fused kernels cover the pixel-decoder shape only: 32 channels per head, L*P in {4, 8, 12, 16}, 2-d
    reference points shared by the batch or per image; fp32, or -- what torch.autocast hands the module -- a bf16 /
    fp16 value with sampling_offsets and attn_logits of the same type and fp32 reference points."""
    if not (isinstance(value, torch.Tensor) and value.is_cuda):
        return False
    if value.dtype in _FUSED_MIXED_FWD:
        if not (sampling_offsets.dtype == attn_logits.dtype == value.dtype
                and reference_points.dtype == torch.float32):
            return False
    elif value.dtype != torch.float32:
        return False
    if value.dim() != 4 or value.size(3) != 32 or sampling_offsets.dim() != 6:
        return False
    L, P = sampling_offsets.size(3), sampling_offsets.size(4)
    if L * P not in (4, 8, 12, 16) or value.size(1) * value.size(2) * 8 >= 0x7fffffff:
        return False
    return (reference_points.dim() == 4 and reference_points.size(-1) == 2
            and reference_points.size(0) in (1, value.size(0)))


def _check_fused(value, shapes, lsi, ref, off, logits, extra=()):
    """The fused op's checks: fp32 throughout, or a bf16 / fp16 value with every other tensor but the fp32
    reference points of the same type (the mixed-precision fused op) -> (N, S, M, D, L, Lq, P, ref batch stride)."""
    named = [("value", value), ("spatial_shapes", shapes), ("level_start_index", lsi),
             ("reference_points", ref), ("sampling_offsets", off), ("attn_logits", logits)] + list(extra)
    _require_cuda_contiguous(named)
    mixed = value.dtype in _FUSED_MIXED_FWD
    if mixed:
        for name, t in [("sampling_offsets", off), ("attn_logits", logits)] + list(extra):
            if t.dtype != value.dtype:
                raise RuntimeError(f"fused MSDA: {name} is {t.dtype} but value is {value.dtype} (the mixed-precision "
                                   "fused op takes one 16-bit type)")
        if ref.dtype != torch.float32:
            raise RuntimeError(f"fused MSDA: reference_points must be float32, found {ref.dtype}")
    if not fused_supported(value, ref, off, logits):
        raise RuntimeError("fused MSDA covers fp32 or bf16 / fp16 (with fp32 reference points), 32 channels per "
                           "head, L*P in {4,8,12,16}, 2-d reference points only; compose the unfused op for other "
                           "shapes")
    N, S, M, D = value.shape
    _, Lq, _, L, P, _ = off.shape
    if tuple(off.shape) != (N, Lq, M, L, P, 2) or logits.numel() != N * Lq * M * L * P \
            or tuple(ref.shape[1:]) != (Lq, L, 2) or shapes.size(0) != L:
        raise RuntimeError("inconsistent shapes for fused MSDA")
    if not mixed:
        for name, t in [("reference_points", ref), ("sampling_offsets", off), ("attn_logits", logits)] + list(extra):
            if t.dtype != torch.float32:
                raise RuntimeError(f"fused MSDA is float32 only: {name} is {t.dtype}")
    ref_stride = 0 if ref.size(0) == 1 and N > 1 else Lq * L * 2
    return N, S, M, D, L, Lq, P, ref_stride


def ms_deform_attn_fused_forward(value, spatial_shapes, level_start_index, reference_points,
                                 sampling_offsets, attn_logits):
    """output [N, Lq, M*D] in value's dtype from raw offsets / logits (msda_b200_fused_forward_strided_f32 on packed
    rows; bf16 / fp16: msda_b200_fused_forward_bf16 / _f16, fp32 arithmetic and one rounding of the output)."""
    N, S, M, D, L, Lq, P, rs = _check_fused(value, spatial_shapes, level_start_index, reference_points,
                                            sampling_offsets, attn_logits)
    if value.dtype in _FUSED_MIXED_FWD:
        with torch.cuda.device(value.device):
            output = torch.empty((N, Lq, M * D), dtype=value.dtype, device=value.device)
            with _timed("forward_mixed"):
                rc = _FUSED_MIXED_FWD[value.dtype](
                    value.data_ptr(), spatial_shapes.data_ptr(), level_start_index.data_ptr(),
                    reference_points.data_ptr(), rs, sampling_offsets.data_ptr(), attn_logits.data_ptr(),
                    N, S, M, D, L, Lq, P, output.data_ptr(), torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, "ms_deform_attn_fused_forward")
        return output
    return _fused_forward("ms_deform_attn_fused_forward", value, spatial_shapes, level_start_index, reference_points,
                          rs, sampling_offsets, 2 * M * L * P, attn_logits, M * L * P, None, None,
                          (N, S, M, D, L, Lq, P))


def _fused_forward(opname, value, shapes, lsi, ref, rs, off, off_stride, logits, logit_stride, off_table, logit_table,
                   dims):
    """msda_b200_fused_forward_strided_f32 on checked tensors; ``off`` / ``logits`` rows ``off_stride`` /
    ``logit_stride`` floats apart, ``off_table`` / ``logit_table`` (both or neither) the per-query additive tables."""
    N, S, M, D, L, Lq, P = dims
    with torch.cuda.device(value.device):
        output = torch.empty((N, Lq, M * D), dtype=value.dtype, device=value.device)
        with _timed("forward"):
            rc = _lib.lib.msda_b200_fused_forward_strided_f32(
                value.data_ptr(), shapes.data_ptr(), lsi.data_ptr(), ref.data_ptr(), rs, off.data_ptr(), off_stride,
                logits.data_ptr(), logit_stride, _ptr(off_table), _ptr(logit_table), N, S, M, D, L, Lq, P,
                output.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, opname)
    return output


def ms_deform_attn_fused_forward_packed(value, spatial_shapes, level_start_index, reference_points,
                                        projections, n_levels, n_points, query_table=None):
    """The fused forward reading the raw offsets and logits in place from ONE projection output
    ``projections`` [N, Lq, 3*M*L*P] = [sampling_offsets (2*M*L*P) | attn_logits (M*L*P)] per query -- the
    stacked ``sampling_offsets`` / ``attention_weights`` Linear (ops/modules/ms_deform_attn.py:105-106) run
    as one GEMM (msda_b200_fused_forward_strided_f32).  ``query_table`` [Lq, 3*M*L*P] (optional) is added to
    the rows of every image inside the kernel: the part of the projection that depends on the query's
    position only (``pos @ W^T + b`` when the projection input is ``src + pos``).  Inference only."""
    N, S, M, D = value.shape
    L, P = int(n_levels), int(n_points)
    width = 3 * M * L * P
    if projections.dim() != 3 or projections.size(0) != N or projections.size(2) != width:
        raise RuntimeError(f"projections must be [N, Lq, {width}]")
    Lq = projections.size(1)
    off = projections[..., :2 * M * L * P]
    logits = projections[..., 2 * M * L * P:]
    named = [("value", value), ("spatial_shapes", spatial_shapes), ("level_start_index", level_start_index),
             ("reference_points", reference_points), ("projections", projections)]
    if query_table is not None:
        named.append(("query_table", query_table))
        if tuple(query_table.shape) != (Lq, width) or query_table.dtype != torch.float32:
            raise RuntimeError(f"query_table must be a float32 [Lq, {width}] tensor")
    _require_cuda_contiguous(named)
    if not fused_supported(value, reference_points, off.view(N, Lq, M, L, P, 2), logits) \
            or tuple(reference_points.shape[1:]) != (Lq, L, 2) or spatial_shapes.size(0) != L \
            or projections.dtype != torch.float32 or reference_points.dtype != torch.float32:
        raise RuntimeError("fused MSDA covers fp32, 32 channels per head, L*P in {4,8,12,16}, 2-d "
                           "reference points only; compose the unfused op for other shapes")
    rs = 0 if reference_points.size(0) == 1 and N > 1 else Lq * L * 2
    return _fused_forward("ms_deform_attn_fused_forward_packed", value, spatial_shapes, level_start_index,
                          reference_points, rs, off, width, logits, width, query_table,
                          query_table[:, 2 * M * L * P:] if query_table is not None else None, (N, S, M, D, L, Lq, P))


_FUSED_MIXED_FWD_STRIDED = {torch.bfloat16: _lib.lib.msda_b200_fused_forward_strided_bf16,
                            torch.float16: _lib.lib.msda_b200_fused_forward_strided_f16}


def ms_deform_attn_fused_mixed_forward_packed_supported(value, reference_points, projections, n_levels, n_points,
                                                        query_table=None) -> bool:
    """Whether ``ms_deform_attn_fused_mixed_forward_packed`` covers these tensors: what the 16-bit fused forward
    covers (``fused_supported``), ``projections`` a contiguous [N, Lq, 3*M*L*P] tensor of value's 16-bit type,
    4-byte aligned, fp32 reference points with Lq rows, and ``query_table`` None or a contiguous fp32 [Lq, 3*M*L*P]
    tensor, 8-byte aligned, on value's device."""
    if not (isinstance(value, torch.Tensor) and value.is_cuda and value.dtype in _FUSED_MIXED_FWD_STRIDED
            and value.dim() == 4 and isinstance(projections, torch.Tensor) and projections.dim() == 3):
        return False
    N, S, M, D = value.shape
    L, P = int(n_levels), int(n_points)
    width = 3 * M * L * P
    if not (projections.dtype == value.dtype and projections.size(0) == N and projections.size(2) == width
            and projections.is_contiguous() and projections.device == value.device and projections.data_ptr() % 4 == 0
            and value.is_contiguous() and value.data_ptr() % 16 == 0):
        return False
    Lq = projections.size(1)
    if query_table is not None and not (
            isinstance(query_table, torch.Tensor) and query_table.dtype == torch.float32
            and tuple(query_table.shape) == (Lq, width) and query_table.is_contiguous()
            and query_table.device == value.device and query_table.data_ptr() % 8 == 0):
        return False
    off = projections[..., :2 * M * L * P]
    return (isinstance(reference_points, torch.Tensor) and reference_points.dtype == torch.float32
            and reference_points.is_contiguous() and reference_points.device == value.device
            and fused_supported(value, reference_points, off.view(N, Lq, M, L, P, 2), projections[..., 2 * M * L * P:])
            and tuple(reference_points.shape[1:]) == (Lq, L, 2))


def ms_deform_attn_fused_mixed_forward_packed(value, spatial_shapes, level_start_index, reference_points,
                                              projections, n_levels, n_points, query_table=None):
    """``ms_deform_attn_fused_forward_packed`` for mixed precision: a bf16 / fp16 ``value`` and ``projections``
    [N, Lq, 3*M*L*P] (the stacked query GEMM run under torch.autocast), fp32 ``reference_points`` and fp32
    ``query_table`` [Lq, 3*M*L*P] (optional).  Each raw offset / logit is widened, then gets its table entry added in
    fp32; output [N, Lq, M*D] in value's dtype is the fp32 strided forward on the widened inputs rounded once
    (msda_b200_fused_forward_strided_bf16 / _f16).  Inference only."""
    N, S, M, D = value.shape
    L, P = int(n_levels), int(n_points)
    named = [("value", value), ("spatial_shapes", spatial_shapes), ("level_start_index", level_start_index),
             ("reference_points", reference_points), ("projections", projections)]
    if query_table is not None:
        named.append(("query_table", query_table))
    _require_cuda_contiguous(named)
    if not ms_deform_attn_fused_mixed_forward_packed_supported(value, reference_points, projections, L, P, query_table) \
            or spatial_shapes.size(0) != L:
        raise RuntimeError("ms_deform_attn_fused_mixed_forward_packed covers a bf16 / fp16 value and projections "
                           "[N, Lq, 3*M*L*P] of the same type, fp32 reference points and query_table [Lq, 3*M*L*P], "
                           "32 channels per head, L*P in {4,8,12,16}")
    Lq = projections.size(1)
    width = 3 * M * L * P
    rs = 0 if reference_points.size(0) == 1 and N > 1 else Lq * L * 2
    with torch.cuda.device(value.device):
        output = torch.empty((N, Lq, M * D), dtype=value.dtype, device=value.device)
        with _timed("forward_mixed"):
            rc = _FUSED_MIXED_FWD_STRIDED[value.dtype](
                value.data_ptr(), spatial_shapes.data_ptr(), level_start_index.data_ptr(), reference_points.data_ptr(),
                rs, projections.data_ptr(), width, projections.data_ptr() + 2 * M * L * P * projections.element_size(),
                width, _ptr(query_table),
                query_table.data_ptr() + 2 * M * L * P * 4 if query_table is not None else None,
                N, S, M, D, L, Lq, P, output.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "ms_deform_attn_fused_mixed_forward_packed")
    return output


def ms_deform_attn_fused_backward(value, spatial_shapes, level_start_index, reference_points,
                                  sampling_offsets, attn_logits, grad_output):
    """[grad_value, grad_sampling_offsets, grad_attn_logits] in the inputs' dtypes (msda_b200_fused_backward_f32;
    bf16 / fp16: msda_b200_fused_backward_bf16 / _f16, grad_value reduced in an fp32 buffer allocated here and
    rounded once, as in ms_deform_attn_mixed_backward)."""
    N, S, M, D, L, Lq, P, rs = _check_fused(value, spatial_shapes, level_start_index, reference_points,
                                            sampling_offsets, attn_logits, [("grad_output", grad_output)])
    if value.dtype in _FUSED_MIXED_FWD:
        if _deterministic():
            return _backward_deterministic(_FUSED_MIXED_BWD_DET[value.dtype],
                                           "ms_deform_attn_fused_backward (deterministic)", value, spatial_shapes,
                                           level_start_index, (sampling_offsets, attn_logits), grad_output,
                                           (N, S, M, D, L, Lq, P), reference_points, rs, kind="backward_mixed")
        with torch.cuda.device(value.device):
            accum = torch.zeros((N, S, M, D), dtype=torch.float32, device=value.device)   # fp32 reductions
            grad_value = torch.empty_like(value)            # rounded from accum
            grad_off = torch.empty_like(sampling_offsets)
            grad_logits = torch.empty_like(attn_logits)
            with _timed("backward_mixed"):
                rc = _FUSED_MIXED_BWD[value.dtype](
                    grad_output.data_ptr(), value.data_ptr(), spatial_shapes.data_ptr(),
                    level_start_index.data_ptr(), reference_points.data_ptr(), rs,
                    sampling_offsets.data_ptr(), attn_logits.data_ptr(), N, S, M, D, L, Lq, P,
                    accum.data_ptr(), grad_value.data_ptr(), grad_off.data_ptr(), grad_logits.data_ptr(),
                    torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, "ms_deform_attn_fused_backward")
        return [grad_value, grad_off, grad_logits]
    if _deterministic():
        return _backward_deterministic(_lib.lib.msda_b200_fused_backward_deterministic_f32,
                                       "ms_deform_attn_fused_backward (deterministic)", value, spatial_shapes,
                                       level_start_index, (sampling_offsets, attn_logits), grad_output,
                                       (N, S, M, D, L, Lq, P), reference_points, rs)
    with torch.cuda.device(value.device):
        grad_value = torch.zeros_like(value)
        grad_off = torch.empty_like(sampling_offsets)
        grad_logits = torch.empty_like(attn_logits)
        with _timed("backward"):
            rc = _lib.lib.msda_b200_fused_backward_f32(
                grad_output.data_ptr(), value.data_ptr(), spatial_shapes.data_ptr(),
                level_start_index.data_ptr(), reference_points.data_ptr(), rs,
                sampling_offsets.data_ptr(), attn_logits.data_ptr(), N, S, M, D, L, Lq, P,
                grad_value.data_ptr(), grad_off.data_ptr(), grad_logits.data_ptr(),
                torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "ms_deform_attn_fused_backward")
    return [grad_value, grad_off, grad_logits]


# ----------------------------------------------------------------------------------------------
# fp32 Linear on the tensor cores (SURVEY.md 8f.3): the nn.Linear layers around the op
# (ops/modules/ms_deform_attn.py:62-65, msdeformattn.py:126-130) as an error-compensated 3xTF32 GEMM.
# Inference only (no backward); torch.nn.functional.linear semantics.
# ----------------------------------------------------------------------------------------------
def linear_tf32x3_supported(x, weight) -> bool:
    return (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32
            and weight.dtype == torch.float32 and weight.dim() == 2 and x.size(-1) == weight.size(1)
            and weight.is_contiguous() and weight.device == x.device
            and weight.size(1) % 32 == 0 and weight.size(0) % 4 == 0 and x.numel() > 0)


def split_weight(weight):
    """The split form of a Linear weight that ``linear_tf32x3(..., presplit=...)`` consumes: ``tf32(W)`` followed by
    ``tf32(W - tf32(W))`` as one flat fp32 tensor of 2 * out * in elements (msda_b200_split_weight_f32).  For weights
    that do not change between calls (inference): one launch per Linear instead of two."""
    if not (isinstance(weight, torch.Tensor) and weight.is_cuda and weight.dtype == torch.float32 and weight.dim() == 2
            and weight.is_contiguous() and weight.numel() % 4 == 0 and weight.numel() > 0):
        raise RuntimeError("split_weight needs a contiguous 2-d fp32 CUDA weight")
    out = torch.empty(2 * weight.numel(), dtype=torch.float32, device=weight.device)
    with torch.cuda.device(weight.device):
        rc = _lib.lib.msda_b200_split_weight_f32(weight.data_ptr(), out.data_ptr(), weight.size(0), weight.size(1),
                                                 torch.cuda.current_stream(weight.device).cuda_stream)
    _lib.check(rc, "split_weight")
    return out


def linear_tf32x3(x, weight, bias=None, relu=False, split_weight_in_kernel=False, presplit=None):
    """``F.linear(x, weight, bias)`` (then ``relu`` if set) for fp32 CUDA tensors; ``x`` [..., in],
    ``presplit``: ``split_weight(weight)`` computed earlier -- the GEMM then runs alone (same bits);
    ``weight`` [out, in] with in % 32 == 0 and out % 4 == 0.  Non-finite inputs give non-finite outputs in
    the affected rows, but an infinite input may come out as NaN where F.linear returns +-inf (the
    error-compensated split forms inf - inf and inf * w_lo of either sign).  ``split_weight_in_kernel``: no pre-pass over
    (and no workspace for) the weight -- for a one-shot "weight" such as transposed activations."""
    named = [("x", x), ("weight", weight)] + ([("bias", bias)] if bias is not None else [])
    _require_cuda_contiguous(named)
    for name, t in named:
        if t.dtype != torch.float32:
            raise RuntimeError(f"{name} must be float32")
    if not linear_tf32x3_supported(x, weight) or (bias is not None and bias.shape != (weight.size(0),)):
        raise RuntimeError("linear_tf32x3 needs x [..., in] and weight [out, in] with in % 32 == 0, out % 4 == 0")
    out_f, in_f = weight.shape
    rows = x.numel() // in_f
    y = torch.empty(x.shape[:-1] + (out_f,), dtype=x.dtype, device=x.device)
    if presplit is not None:
        if not (presplit.is_cuda and presplit.device == x.device and presplit.dtype == torch.float32
                and presplit.is_contiguous() and presplit.numel() == 2 * out_f * in_f):
            raise RuntimeError("presplit must be split_weight(weight) on x's device")
        fn = (_lib.lib.msda_b200_linear_presplit_deterministic_f32 if _deterministic()
              else _lib.lib.msda_b200_linear_presplit_f32)
        with torch.cuda.device(x.device):
            rc = fn(x.data_ptr(), presplit.data_ptr(),
                                                        bias.data_ptr() if bias is not None else None, y.data_ptr(),
                                                        rows, out_f, in_f, 1 if relu else 0,
                                                        torch.cuda.current_stream(x.device).cuda_stream)
        _lib.check(rc, "linear_tf32x3")
        return y
    workspace = None if split_weight_in_kernel else \
        torch.empty(2 * out_f * in_f, dtype=torch.float32, device=x.device)
    fn = _lib.lib.msda_b200_linear_deterministic_f32 if _deterministic() else _lib.lib.msda_b200_linear_f32
    with torch.cuda.device(x.device):
        rc = fn(x.data_ptr(), weight.data_ptr(),
                                           bias.data_ptr() if bias is not None else None, y.data_ptr(),
                                           rows, out_f, in_f, 1 if relu else 0,
                                           workspace.data_ptr() if workspace is not None else None,
                                           torch.cuda.current_stream(x.device).cuda_stream)
    _lib.check(rc, "linear_tf32x3")
    return y


def add_layernorm_supported(x, residual, weight, bias=None, need_bias=False) -> bool:
    """Whether the fused residual + LayerNorm kernels cover these tensors; callers pass the norm's bias
    with need_bias=True so that an nn.LayerNorm(bias=False), or affine parameters that are not
    contiguous fp32 tensors on x's device, take torch's own path."""
    def affine_ok(t):
        return (isinstance(t, torch.Tensor) and t.dtype == torch.float32 and t.is_contiguous()
                and t.device == x.device and t.numel() == x.size(-1))
    return (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.is_contiguous()
            and x.size(-1) in (128, 256, 384, 512) and x.numel() > 0 and affine_ok(weight)
            and (affine_ok(bias) if (need_bias or bias is not None) else True)
            and (residual is None or (residual.shape == x.shape and residual.is_contiguous()
                                      and residual.dtype == torch.float32 and residual.device == x.device)))


def add_layernorm(x, residual, weight, bias, eps=1e-5):
    """``F.layer_norm(x + residual, (C,), weight, bias, eps)`` in one pass (fp32 CUDA, C in {128,...,512});
    ``residual`` may be None.  Inference only (no backward)."""
    if not x.is_cuda:
        raise RuntimeError("Not implemented on the CPU")
    if not add_layernorm_supported(x, residual, weight) or bias is None or bias.shape != weight.shape:
        raise RuntimeError("add_layernorm needs contiguous fp32 CUDA tensors with a last dimension of "
                           "128, 256, 384 or 512 and affine parameters")
    y = torch.empty_like(x)
    cols = x.size(-1)
    with torch.cuda.device(x.device):
        rc = _lib.lib.msda_b200_add_layernorm_f32(
            x.data_ptr(), residual.data_ptr() if residual is not None else None, weight.data_ptr(),
            bias.data_ptr(), y.data_ptr(), x.numel() // cols, cols, float(eps),
            torch.cuda.current_stream(x.device).cuda_stream)
    _lib.check(rc, "add_layernorm")
    return y


# ---------------------------------------------------------------- mixed precision (torch.autocast) residual + LayerNorm
_LN_MIXED = {torch.bfloat16: _lib.lib.msda_b200_add_layernorm_mixed_bf16,
             torch.float16: _lib.lib.msda_b200_add_layernorm_mixed_f16}
_LN_MIXED_BWD = {torch.bfloat16: _lib.lib.msda_b200_add_layernorm_mixed_backward_bf16,
                 torch.float16: _lib.lib.msda_b200_add_layernorm_mixed_backward_f16}
_LN_MIXED_BWD_DET = {torch.bfloat16: _lib.lib.msda_b200_add_layernorm_mixed_backward_deterministic_bf16,
                     torch.float16: _lib.lib.msda_b200_add_layernorm_mixed_backward_deterministic_f16}


def _rows16_ok(t, x) -> bool:
    """`t` a contiguous bf16 / fp16 tensor shaped like `x` on x's device, 8-byte aligned (the kernels' 4-element
    accesses)."""
    return (isinstance(t, torch.Tensor) and t.dtype in _LN_MIXED and t.shape == x.shape and t.is_contiguous()
            and t.device == x.device and t.data_ptr() % 8 == 0)


def add_layernorm_mixed_supported(x, residual, weight, bias=None, need_bias=False) -> bool:
    """Whether the mixed-precision residual + LayerNorm kernels cover these tensors: ``x`` what ``add_layernorm``
    takes and 16-byte aligned, ``residual`` a contiguous bf16 / fp16 tensor of x's shape, 8-byte aligned (an unaligned
    view takes torch's path in the modules)."""
    return (add_layernorm_supported(x, None, weight, bias, need_bias) and x.data_ptr() % 16 == 0
            and weight.data_ptr() % 16 == 0 and (bias is None or bias.data_ptr() % 16 == 0)
            and _rows16_ok(residual, x))


def add_layernorm_mixed(x, residual, weight, bias, eps=1e-5, want_y16=True):
    """``(y, y16)``: ``y = F.layer_norm(x + residual.float(), (C,), weight, bias, eps)`` (fp32, bit-identical to
    ``add_layernorm(x, residual.float(), ...)``) and ``y16 = y.to(residual.dtype)`` (None unless ``want_y16``), for an
    fp32 ``x`` and a bf16 / fp16 ``residual`` -- torch.autocast's ``layer_norm(x + sublayer)`` and the cast of its
    result for the next GEMM, in one pass (msda_b200_add_layernorm_mixed_bf16 / _f16).  Inference only (no autograd:
    functions.AddLayerNormMixedFunction)."""
    if not x.is_cuda:
        raise RuntimeError("Not implemented on the CPU")
    if not add_layernorm_mixed_supported(x, residual, weight, bias, need_bias=True):
        raise RuntimeError("add_layernorm_mixed needs a contiguous fp32 CUDA x (16-byte aligned) with a last dimension of "
                           "128, 256, 384 or 512, a contiguous bf16 / fp16 residual of its shape (8-byte aligned) and "
                           "fp32 affine parameters")
    y = torch.empty_like(x)
    y16 = torch.empty_like(residual) if want_y16 else None
    cols = x.size(-1)
    with torch.cuda.device(x.device):
        with _timed("add_layernorm_mixed"):
            rc = _LN_MIXED[residual.dtype](x.data_ptr(), residual.data_ptr(), weight.data_ptr(), bias.data_ptr(),
                                           y.data_ptr(), _ptr(y16), x.numel() // cols, cols, float(eps),
                                           torch.cuda.current_stream(x.device).cuda_stream)
    _lib.check(rc, "add_layernorm_mixed")
    return y, y16


def add_layernorm_mixed_backward_supported(x, residual, weight) -> bool:
    """Whether ``add_layernorm_mixed_backward`` covers these tensors: those of ``add_layernorm_mixed_supported`` with a
    last dimension of 128 or 256."""
    return add_layernorm_mixed_supported(x, residual, weight) and x.size(-1) in (128, 256)


def add_layernorm_mixed_backward(grad_y, grad_y16, x, residual, weight, eps=1e-5):
    """``(grad_x, grad_residual, grad_weight, grad_bias)`` of ``add_layernorm_mixed`` from the gradients of ``y`` (fp32)
    and ``y16`` (residual's dtype); either may be None.  With ``g = grad_y + grad_y16.float()``, ``grad_x`` (fp32) is
    bit-identical to ``add_layernorm_backward(g, x, residual.float(), weight)[0]`` and ``grad_residual`` is
    ``grad_x.to(residual.dtype)``: what autograd computes for torch.autocast's composition.  With
    torch.use_deterministic_algorithms(True) the deterministic entries (per-CTA partials added in CTA order)."""
    if grad_y is None and grad_y16 is None:
        raise RuntimeError("add_layernorm_mixed_backward needs grad_y or grad_y16")
    if not add_layernorm_mixed_backward_supported(x, residual, weight) \
            or (grad_y is not None and not (grad_y.shape == x.shape and grad_y.is_contiguous()
                                            and grad_y.dtype == torch.float32 and grad_y.device == x.device
                                            and grad_y.data_ptr() % 16 == 0)) \
            or (grad_y16 is not None and not (_rows16_ok(grad_y16, x) and grad_y16.dtype == residual.dtype)):
        raise RuntimeError("add_layernorm_mixed_backward needs what add_layernorm_mixed needs, a last dimension of 128 or "
                           "256, a contiguous fp32 grad_y (16-byte aligned) and a contiguous grad_y16 of residual's "
                           "dtype (8-byte aligned)")
    gx = torch.empty_like(x)
    gr = torch.empty_like(residual)
    gg, gb = torch.empty_like(weight), torch.empty_like(weight)
    cols = x.size(-1)
    rows = x.numel() // cols
    with torch.cuda.device(x.device):
        args = (_ptr(grad_y), _ptr(grad_y16), x.data_ptr(), residual.data_ptr(), weight.data_ptr(), gx.data_ptr(),
                gr.data_ptr(), gg.data_ptr(), gb.data_ptr(), rows, cols, float(eps))
        stream = torch.cuda.current_stream(x.device).cuda_stream
        with _timed("add_layernorm_mixed_backward"):
            if _deterministic():
                ws = _workspace(_lib.lib.msda_b200_add_layernorm_backward_deterministic_workspace_bytes(rows, cols), x)
                rc = _LN_MIXED_BWD_DET[residual.dtype](*args, ws.data_ptr(), stream)
            else:
                rc = _LN_MIXED_BWD[residual.dtype](*args, stream)
    _lib.check(rc, "add_layernorm_mixed_backward")
    return gx, gr, gg, gb


def _vec_ok(t, x) -> bool:
    return (isinstance(t, torch.Tensor) and t.device == x.device and t.dtype == torch.float32 and t.is_contiguous()
            and t.shape == (x.size(1),))


# the GroupNorm maps' element types and the alignment their 4-element accesses need: fp32, or the bf16 / fp16 map a
# convolution writes under torch.autocast (the mixed-precision kernels, DESIGN.md 11.3)
_MAP_ALIGN = {torch.float32: 16, torch.bfloat16: 8, torch.float16: 8}
_GN_MIXED = {dtype: {name: getattr(_lib.lib, f"msda_b200_{name}_{sfx}")
                     for name in ("group_norm_nchw_mixed", "group_norm_nchw_mixed_train", "group_norm_nchw_to_rows_mixed",
                                  "group_norm_nchw_to_rows_mixed_train", "group_norm_backward_nchw_mixed",
                                  "group_norm_rows_backward_mixed", "add_channel_bias_nchw")}
             for dtype, sfx in ((torch.bfloat16, "bf16"), (torch.float16, "f16"))}


def _map_ok(x, weight, bias, groups, up=None) -> bool:
    """What every GroupNorm kernel needs of an NCHW map: x contiguous fp32 (16-byte aligned) or bf16 / fp16 (8-byte
    aligned) on a CUDA device, with H*W a multiple of 4 (the planes are walked 4 elements at a time); weight and bias
    contiguous fp32 [C] on x's device; C divisible by groups; with `up` (the map the forward up-samples and adds): W a
    multiple of 4 as well, and `up` a contiguous fp32 map with x's batch and channels on x's device."""
    return (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype in _MAP_ALIGN and x.dim() == 4
            and x.is_contiguous() and x.numel() > 0 and (x.size(2) * x.size(3)) % 4 == 0
            and x.data_ptr() % _MAP_ALIGN[x.dtype] == 0
            and isinstance(groups, int) and groups > 0 and x.size(1) % groups == 0 and _vec_ok(weight, x)
            and _vec_ok(bias, x)
            and (up is None or (isinstance(up, torch.Tensor) and up.dtype == torch.float32 and up.dim() == 4
                                and up.is_contiguous() and up.device == x.device and up.shape[:2] == x.shape[:2]
                                and x.size(3) % 4 == 0)))


def _rows_view_ok(rows, x) -> bool:
    """What the rows kernels need besides the map: C a multiple of 32, and `rows` an fp32 [N, H*W, C] view on x's device
    with unit channel stride and 16-byte aligned rows (e.g. a level's slice of the concatenated [N, S, C] tensor)."""
    return (x.size(1) % 32 == 0 and isinstance(rows, torch.Tensor) and rows.device == x.device
            and rows.dtype == torch.float32 and rows.dim() == 3
            and tuple(rows.shape) == (x.size(0), x.size(2) * x.size(3), x.size(1)) and rows.stride(2) == 1
            and rows.stride(1) >= x.size(1) and rows.stride(1) % 4 == 0 and rows.stride(0) % 4 == 0
            and rows.data_ptr() % 16 == 0)


def _check_channel_bias(channel_bias, x):
    if channel_bias is not None and not _vec_ok(channel_bias, x):
        raise RuntimeError("channel_bias must be a contiguous fp32 [C] tensor on x's device")


def _check_mean_rstd(mean_rstd, x, groups):
    if not (isinstance(mean_rstd, torch.Tensor) and mean_rstd.device == x.device and mean_rstd.dtype == torch.float32
            and mean_rstd.is_contiguous() and mean_rstd.shape == (x.size(0), groups, 2)):
        raise RuntimeError("mean_rstd must be the contiguous fp32 [N, groups, 2] tensor of the training forward")


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _workspace(nbytes, x):
    return torch.empty(int(nbytes), dtype=torch.uint8, device=x.device)


def group_norm_supported(x, norm, up=None) -> bool:
    """Whether the fused GroupNorm kernels cover `norm(x)` (x: NCHW fp32, bf16 or fp16 CUDA, contiguous; `norm` an
    affine nn.GroupNorm whose parameters are contiguous fp32 [C] tensors on x's device)."""
    return isinstance(norm, torch.nn.GroupNorm) and _map_ok(x, norm.weight, norm.bias, norm.num_groups, up)


def group_norm_rows_supported(x, norm, out_rows) -> bool:
    """Whether `group_norm_rows` covers these tensors: the map as for `group_norm`, channels a multiple of 32, and
    `out_rows` an fp32 [N, H*W, C] view with unit channel stride (a slice of the concatenated [N, S, C] tensor)."""
    return group_norm_supported(x, norm) and _rows_view_ok(out_rows, x)


def _out_dtype(x, out_dtype):
    """The output type of a GroupNorm of `x`: fp32 (None: what F.group_norm returns under torch.autocast), or -- for a
    16-bit x -- x's own type, the rounded copy the next convolution reads."""
    if out_dtype is None or out_dtype == torch.float32 or out_dtype == x.dtype:
        return torch.float32 if out_dtype is None else out_dtype
    raise RuntimeError(f"out_dtype must be None, torch.float32 or the map's dtype {x.dtype}, not {out_dtype}")


def _group_norm_nchw(name, x, weight, bias, groups, eps, relu, up, channel_bias, stats, out_dtype=None):
    """The NCHW forward -> (y, mean_rstd [N, groups, 2] when `stats`, else None); y of type `out_dtype` (None: fp32)."""
    if not _map_ok(x, weight, bias, groups, up):
        raise RuntimeError(f"{name} needs a contiguous NCHW fp32 CUDA map with H*W (and, with `up`, W) a multiple of 4, "
                           "contiguous fp32 [C] weight and bias on the same device, C divisible by groups and, if "
                           "given, a contiguous `up` map with the same batch and channels")
    _check_channel_bias(channel_bias, x)
    out_dtype = _out_dtype(x, out_dtype)
    N, C, H, W = x.shape
    y = torch.empty_like(x, dtype=out_dtype)
    mean_rstd = torch.empty(N, groups, 2, dtype=torch.float32, device=x.device) if stats else None
    with torch.cuda.device(x.device):
        ws = _workspace(_lib.lib.msda_b200_group_norm_workspace_bytes(N, groups), x)
        tail = (N, C, H, W, groups, float(eps), int(bool(relu)), _ptr(up), up.size(2) if up is not None else 0,
                up.size(3) if up is not None else 0, ws.data_ptr(), torch.cuda.current_stream(x.device).cuda_stream)
        if x.dtype == torch.float32:
            head = (x.data_ptr(), _ptr(channel_bias), weight.data_ptr(), bias.data_ptr(), y.data_ptr())
            rc = (_lib.lib.msda_b200_group_norm_nchw_train_f32(*head, mean_rstd.data_ptr(), *tail) if stats
                  else _lib.lib.msda_b200_group_norm_nchw_f32(*head, *tail))
        else:                      # a 16-bit map: the fp32 y or its 16-bit copy y16
            y32, y16 = (y, None) if out_dtype == torch.float32 else (None, y)
            head = (x.data_ptr(), _ptr(channel_bias), weight.data_ptr(), bias.data_ptr(), _ptr(y32), _ptr(y16))
            entries = _GN_MIXED[x.dtype]
            rc = (entries["group_norm_nchw_mixed_train"](*head, mean_rstd.data_ptr(), *tail) if stats
                  else entries["group_norm_nchw_mixed"](*head, *tail))
    _lib.check(rc, name)
    return y, mean_rstd


def _group_norm_rows(name, x, weight, bias, groups, eps, out_rows, channel_bias, relu, stats):
    """The rows forward: writes out_rows -> mean_rstd [N, groups, 2] when `stats`, else None."""
    if not (_map_ok(x, weight, bias, groups) and _rows_view_ok(out_rows, x)):
        raise RuntimeError(f"{name} needs what group_norm needs, channels % 32 == 0 and an fp32 [N, H*W, C] "
                           "destination view with unit channel stride on the same device")
    _check_channel_bias(channel_bias, x)
    N, C, H, W = x.shape
    mean_rstd = torch.empty(N, groups, 2, dtype=torch.float32, device=x.device) if stats else None
    with torch.cuda.device(x.device):
        ws = _workspace(_lib.lib.msda_b200_group_norm_workspace_bytes(N, groups), x)
        head = (x.data_ptr(), _ptr(channel_bias), weight.data_ptr(), bias.data_ptr(), out_rows.data_ptr())
        tail = (out_rows.stride(1), out_rows.stride(0), N, C, H * W, groups, float(eps), int(bool(relu)), ws.data_ptr(),
                torch.cuda.current_stream(x.device).cuda_stream)
        if x.dtype == torch.float32:
            rc = (_lib.lib.msda_b200_group_norm_nchw_to_rows_train_f32(*head, mean_rstd.data_ptr(), *tail) if stats
                  else _lib.lib.msda_b200_group_norm_nchw_to_rows_f32(*head, *tail))
        else:                      # a 16-bit map, fp32 rows
            entries = _GN_MIXED[x.dtype]
            rc = (entries["group_norm_nchw_to_rows_mixed_train"](*head, mean_rstd.data_ptr(), *tail) if stats
                  else entries["group_norm_nchw_to_rows_mixed"](*head, *tail))
    _lib.check(rc, name)
    return mean_rstd


def group_norm(x, norm, relu=False, up=None, channel_bias=None, out_dtype=None):
    """``norm(x)`` (``norm(x + channel_bias[None, :, None, None])`` when the producing convolution ran without
    its bias) for an ``nn.GroupNorm`` on an NCHW fp32 CUDA map, optionally followed by ReLU and by
    ``+ F.interpolate(up, size=x.shape[-2:], mode="bilinear", align_corners=False)`` -- the epilogues of the
    pixel decoder's input projections and FPN level (msdeformattn.py:233-248, :369-379) -- in two passes
    over x (statistics, apply) instead of torch's four to six kernels.  No autograd: training goes through
    functions.GroupNormFunction (group_norm_train / group_norm_backward).

    A bf16 / fp16 ``x`` (a convolution's output under torch.autocast) is widened on load; ``up``, the affine
    parameters and ``channel_bias`` stay fp32.  The result is fp32 (``out_dtype`` None: what torch.autocast's
    ``F.group_norm(x.float(), ...)`` composition returns), bit-identical to the fp32 kernels on ``x.float()``; with
    ``out_dtype=x.dtype`` it is that result rounded to x's type, the copy the next convolution reads."""
    return _group_norm_nchw("group_norm", x, norm.weight, norm.bias, norm.num_groups, norm.eps, relu, up, channel_bias,
                            False, out_dtype)[0]


def group_norm_rows(x, norm, out_rows, channel_bias=None, relu=False):
    """``out_rows[n, p, c] = norm(x + channel_bias)[n, c, p]`` (p = flattened pixel): GroupNorm of an NCHW map written
    straight into the ``[N, pixels, C]`` layout of the deformable encoder (``src.flatten(2).transpose(1, 2)``),
    e.g. into the level's rows of the concatenated tensor.  No autograd: training goes through
    functions.GroupNormRowsFunction (group_norm_rows_train / group_norm_rows_backward).  Returns out_rows.  x may be
    bf16 / fp16 (widened on load); out_rows is fp32."""
    _group_norm_rows("group_norm_rows", x, norm.weight, norm.bias, norm.num_groups, norm.eps, out_rows, channel_bias,
                     relu, False)
    return out_rows


def channel_bias_supported(x, bias) -> bool:
    # the map predicate with the bias in the place of both affine parameters (one group)
    return _map_ok(x, bias, bias, 1)


def add_channel_bias_(x, bias):
    """``x += bias[None, :, None, None]`` in place on a contiguous NCHW fp32 CUDA map (the bias of a convolution
    that ran without one: torch's own broadcast add runs at less than half of the memory roofline).  A bf16 / fp16
    map with the fp32 bias: ``x.copy_((x.float() + bias).to(x.dtype))``, one rounding per element."""
    if not channel_bias_supported(x, bias):
        raise RuntimeError("add_channel_bias_ needs a contiguous NCHW fp32 CUDA map with H*W % 4 == 0 and a [C] bias")
    entry = (_lib.lib.msda_b200_add_channel_bias_nchw_f32 if x.dtype == torch.float32
             else _GN_MIXED[x.dtype]["add_channel_bias_nchw"])
    with torch.cuda.device(x.device):
        rc = entry(x.data_ptr(), bias.data_ptr(), x.size(0), x.size(1), x.size(2) * x.size(3),
                   torch.cuda.current_stream(x.device).cuda_stream)
    _lib.check(rc, "add_channel_bias_")
    return x


def transpose2d(x, out=None):
    """``x.t().contiguous()`` for a contiguous fp32 CUDA matrix (operand preparation for the weight-gradient GEMM;
    the [pixels, C] -> [C, pixels] turn of the encoder memory); ``out``: a contiguous [cols, rows] destination."""
    if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.is_contiguous() and x.numel() > 0):
        raise RuntimeError("transpose2d needs a contiguous 2-d fp32 CUDA tensor")
    if out is not None and not (out.is_cuda and out.device == x.device and out.dtype == torch.float32
                                and out.is_contiguous() and out.numel() == x.numel()):
        raise RuntimeError("transpose2d: out must be a contiguous fp32 tensor of x's size on x's device")
    y = torch.empty(x.size(1), x.size(0), dtype=x.dtype, device=x.device) if out is None else out
    with torch.cuda.device(x.device):
        rc = _lib.lib.msda_b200_transpose_f32(x.data_ptr(), y.data_ptr(), x.size(0), x.size(1),
                                              torch.cuda.current_stream(x.device).cuda_stream)
    _lib.check(rc, "transpose2d")
    return y


def linear_wgrad_supported(grad_y, x) -> bool:
    return (isinstance(grad_y, torch.Tensor) and grad_y.is_cuda and grad_y.dtype == torch.float32 and x.dtype == torch.float32
            and grad_y.dim() == 2 and x.dim() == 2 and grad_y.size(0) == x.size(0) and grad_y.numel() > 0 and x.numel() > 0
            and grad_y.is_contiguous() and x.is_contiguous() and grad_y.size(1) % 4 == 0 and x.size(1) % 4 == 0
            and x.device == grad_y.device)


def linear_wgrad(grad_y, x, with_bias=True):
    """(grad_weight [out, in], grad_bias [out] or None) of ``F.linear`` from ``grad_y`` [rows, out] and ``x``
    [rows, in] (contiguous fp32 CUDA): grad_y^T @ x and the column sums of grad_y in one kernel."""
    if not grad_y.is_cuda:
        raise RuntimeError("Not implemented on the CPU")
    if not linear_wgrad_supported(grad_y, x):
        raise RuntimeError("linear_wgrad needs contiguous fp32 CUDA matrices grad_y [rows, out], x [rows, in] with "
                           "out % 4 == 0 and in % 4 == 0")
    gw = torch.empty(grad_y.size(1), x.size(1), dtype=torch.float32, device=x.device)
    gb = torch.empty(grad_y.size(1), dtype=torch.float32, device=x.device) if with_bias else None
    rows, out_f, in_f = grad_y.size(0), grad_y.size(1), x.size(1)
    with torch.cuda.device(x.device):
        stream = torch.cuda.current_stream(x.device).cuda_stream
        if _deterministic():      # per-chunk partial tiles, added in chunk order
            ws = _workspace(_lib.lib.msda_b200_linear_wgrad_deterministic_workspace_bytes(rows, out_f, in_f), x)
            rc = _lib.lib.msda_b200_linear_wgrad_deterministic_f32(grad_y.data_ptr(), x.data_ptr(), gw.data_ptr(),
                                                                   _ptr(gb), rows, out_f, in_f, ws.data_ptr(), stream)
        else:
            rc = _lib.lib.msda_b200_linear_wgrad_f32(grad_y.data_ptr(), x.data_ptr(), gw.data_ptr(), _ptr(gb), rows,
                                                     out_f, in_f, stream)
    _lib.check(rc, "linear_wgrad")
    return gw, gb


# ---------------------------------------------------------------- 16-bit Linear under torch.autocast (DESIGN.md 11.4)
_LIN_MIXED = {torch.bfloat16: _lib.lib.msda_b200_linear_mixed_bf16, torch.float16: _lib.lib.msda_b200_linear_mixed_f16}
_LIN_MIXED_WGRAD = {torch.bfloat16: _lib.lib.msda_b200_linear_mixed_wgrad_bf16,
                    torch.float16: _lib.lib.msda_b200_linear_mixed_wgrad_f16}


def _mat16_ok(t, dtype, device) -> bool:
    """`t` a contiguous tensor of `dtype` on `device` whose data is 16-byte aligned (the kernels' TMA loads)."""
    return (isinstance(t, torch.Tensor) and t.dtype == dtype and t.device == device and t.is_contiguous()
            and t.numel() > 0 and t.data_ptr() % 16 == 0)


def linear_mixed_shapes_supported(x, out_features, in_features, bias=None) -> bool:
    """Whether the 16-bit GEMM covers ``x`` [..., in_features] -> [..., out_features]: x a contiguous 16-byte aligned
    bf16 / fp16 CUDA tensor, in % 8 == 0 and out % 8 == 0; ``bias`` None or a contiguous fp32 [out] on x's device."""
    return (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype in _LIN_MIXED and x.dim() >= 1
            and _mat16_ok(x, x.dtype, x.device) and x.size(-1) == in_features
            and out_features % 8 == 0 and in_features % 8 == 0 and x.numel() // in_features < 2 ** 31
            and (bias is None or (isinstance(bias, torch.Tensor) and bias.dtype == torch.float32
                                  and bias.device == x.device and bias.is_contiguous()
                                  and tuple(bias.shape) == (out_features,))))


def linear_mixed_supported(x, weight16, bias=None) -> bool:
    """Whether ``linear_mixed`` covers these tensors: ``x`` [..., in] a contiguous bf16 / fp16 CUDA tensor and
    ``weight16`` [out, in] a contiguous one of x's dtype, both 16-byte aligned, with in % 8 == 0 and out % 8 == 0;
    ``bias`` None or a contiguous fp32 [out] tensor on x's device."""
    return (isinstance(weight16, torch.Tensor) and weight16.dim() == 2 and isinstance(x, torch.Tensor)
            and _mat16_ok(weight16, x.dtype, x.device)
            and linear_mixed_shapes_supported(x, weight16.size(0), weight16.size(1), bias))


def linear_mixed_preferred(rows, out_features, in_features, relu, op) -> bool:
    """Whether the 16-bit kernel is measured at least as fast as torch's 16-bit GEMM for `op` ("forward" or
    "input_gradient") of a Linear with these shapes (NVIDIA B200, profiles/r9_linear_mixed.jsonl, DESIGN.md 11.4):
    * the input gradient is 4-29 % slower than cuBLAS at every measured site (in_features = 256 with out_features
      96 ... 1024, 172 032 and 344 064 rows);
    * the forward is faster or level everywhere except in = out = 256 without ReLU above 262 144 rows (0.076 against
      0.071 ms at 344 064 rows; 0.046 against 0.048 ms at 172 032).
    Callers take torch's GEMM where this is False, unless determinism is asked for."""
    if op == "input_gradient":
        return False
    if op == "forward":
        return not (in_features == out_features == 256 and not relu and rows > 262144)
    raise ValueError(f"unknown op {op!r}")


def linear_mixed(x, weight16, bias=None, relu=False):
    """``F.linear(x, weight16, bias)`` (then ReLU if ``relu``) as torch.autocast computes it, for a bf16 / fp16 ``x``
    and ``weight16`` of one type and an fp32 ``bias``: the bias is added to the fp32 accumulator and the result rounded
    once to x's dtype (msda_b200_linear_mixed_bf16 / _f16).  Also the input gradient ``grad_y @ weight16`` with the
    transposed weight.  Inference only (no autograd: functions.LinearMixedFunction)."""
    if not isinstance(x, torch.Tensor) or not x.is_cuda:
        raise RuntimeError("Not implemented on the CPU")
    if not linear_mixed_supported(x, weight16, bias):
        raise RuntimeError("linear_mixed needs contiguous 16-byte aligned bf16 / fp16 CUDA tensors x [..., in] and "
                           "weight16 [out, in] of one dtype with in % 8 == 0 and out % 8 == 0, and an fp32 bias [out] "
                           "or None")
    out_f, in_f = weight16.shape
    y = torch.empty(x.shape[:-1] + (out_f,), dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device):
        with _timed("linear_mixed"):
            rc = _LIN_MIXED[x.dtype](x.data_ptr(), weight16.data_ptr(), _ptr(bias), y.data_ptr(), x.numel() // in_f,
                                     out_f, in_f, 1 if relu else 0, torch.cuda.current_stream(x.device).cuda_stream)
    _lib.check(rc, "linear_mixed")
    return y


def linear_mixed_wgrad_supported(grad_y, x) -> bool:
    """Whether ``linear_mixed_wgrad`` covers these tensors: contiguous 16-byte aligned bf16 / fp16 CUDA matrices
    ``grad_y`` [rows, out] and ``x`` [rows, in] of one dtype, out % 8 == 0 and in % 8 == 0."""
    return (isinstance(grad_y, torch.Tensor) and grad_y.is_cuda and grad_y.dtype in _LIN_MIXED_WGRAD
            and grad_y.dim() == 2 and isinstance(x, torch.Tensor) and x.dim() == 2 and grad_y.size(0) == x.size(0)
            and _mat16_ok(grad_y, grad_y.dtype, grad_y.device) and _mat16_ok(x, grad_y.dtype, grad_y.device)
            and grad_y.size(1) % 8 == 0 and x.size(1) % 8 == 0 and grad_y.size(0) < 2 ** 31)


def linear_mixed_wgrad(grad_y, x, with_bias=True):
    """(grad_weight [out, in], grad_bias [out] or None), both fp32, of ``F.linear`` from 16-bit ``grad_y`` [rows, out]
    and ``x`` [rows, in]: grad_y^T @ x and the column sums of grad_y with fp32 accumulation, never rounded to 16 bits.
    Deterministic by construction (per-chunk partials in a workspace, added in chunk order by a second launch)."""
    if not isinstance(grad_y, torch.Tensor) or not grad_y.is_cuda:
        raise RuntimeError("Not implemented on the CPU")
    if not linear_mixed_wgrad_supported(grad_y, x):
        raise RuntimeError("linear_mixed_wgrad needs contiguous 16-byte aligned bf16 / fp16 CUDA matrices grad_y "
                           "[rows, out] and x [rows, in] of one dtype with out % 8 == 0 and in % 8 == 0")
    rows, out_f, in_f = grad_y.size(0), grad_y.size(1), x.size(1)
    gw = torch.empty(out_f, in_f, dtype=torch.float32, device=x.device)
    gb = torch.empty(out_f, dtype=torch.float32, device=x.device) if with_bias else None
    with torch.cuda.device(x.device):
        ws = _workspace(_lib.lib.msda_b200_linear_mixed_wgrad_workspace_bytes(rows, out_f, in_f), x)
        with _timed("linear_mixed_wgrad"):
            rc = _LIN_MIXED_WGRAD[grad_y.dtype](grad_y.data_ptr(), x.data_ptr(), gw.data_ptr(), _ptr(gb), rows, out_f,
                                                in_f, ws.data_ptr(), torch.cuda.current_stream(x.device).cuda_stream)
    _lib.check(rc, "linear_mixed_wgrad")
    return gw, gb


def add_layernorm_backward(grad_y, x, residual, weight, eps=1e-5):
    """(grad_v, grad_weight, grad_bias) of ``layer_norm(x + residual)``; grad_v is the gradient of both x and
    residual.  Last dimension 128 or 256."""
    if not (add_layernorm_supported(x, residual, weight) and x.size(-1) in (128, 256)
            and grad_y.shape == x.shape and grad_y.is_contiguous() and grad_y.dtype == torch.float32):
        raise RuntimeError("add_layernorm_backward needs contiguous fp32 CUDA tensors with a last dimension of 128 or 256")
    gv = torch.empty_like(x)
    gg, gb = torch.empty_like(weight), torch.empty_like(weight)
    cols = x.size(-1)
    rows = x.numel() // cols
    with torch.cuda.device(x.device):
        args = (grad_y.data_ptr(), x.data_ptr(), _ptr(residual), weight.data_ptr(), gv.data_ptr(), gg.data_ptr(),
                gb.data_ptr(), rows, cols, float(eps))
        stream = torch.cuda.current_stream(x.device).cuda_stream
        if _deterministic():      # per-CTA partials of grad_weight / grad_bias, added in CTA order
            ws = _workspace(_lib.lib.msda_b200_add_layernorm_backward_deterministic_workspace_bytes(rows, cols), x)
            rc = _lib.lib.msda_b200_add_layernorm_backward_deterministic_f32(*args, ws.data_ptr(), stream)
        else:
            rc = _lib.lib.msda_b200_add_layernorm_backward_f32(*args, stream)
    _lib.check(rc, "add_layernorm_backward")
    return gv, gg, gb


# ---------------------------------------------------------------- GroupNorm training (forward + backward)
def group_norm_train(x, weight, bias, groups, eps, relu=False, up=None, channel_bias=None, out_dtype=None):
    """Training forward of ``group_norm``: ``(y, mean_rstd)`` with ``y`` bit-identical to ``group_norm`` on the same
    inputs and ``mean_rstd`` [N, groups, 2] the (mean, rstd) of ``x + channel_bias`` that the backward needs.  The
    affine parameters are passed as tensors (weight, bias [C]) so that autograd can follow them."""
    return _group_norm_nchw("group_norm_train", x, weight, bias, groups, eps, relu, up, channel_bias, True, out_dtype)


def group_norm_rows_train(x, weight, bias, groups, eps, out_rows, channel_bias=None, relu=False):
    """Training forward of ``group_norm_rows``: writes ``out_rows`` (bit-identical to ``group_norm_rows``) and returns
    ``mean_rstd`` [N, groups, 2]."""
    return _group_norm_rows("group_norm_rows_train", x, weight, bias, groups, eps, out_rows, channel_bias, relu, True)


def group_norm_backward(grad_y, x, weight, bias, mean_rstd, groups, relu=False, channel_bias=None, up_shape=None,
                        with_channel_bias=False):
    """Gradients of ``group_norm_train``: ``(grad_x, grad_weight, grad_bias, grad_channel_bias, grad_up)`` from
    ``grad_y`` and the forward's inputs and ``mean_rstd``.  ``grad_channel_bias`` is computed when
    ``with_channel_bias`` (else None); ``grad_up`` [N, C, *up_shape] when ``up_shape`` (the up-sampled map's (h, w))
    is given (else None).  Three launches, four with ``grad_up``; deterministic.  For a bf16 / fp16 ``x``, ``grad_y``
    is fp32 or of x's type (the gradient of whichever output the forward returned) and ``grad_x`` is of x's type: the
    fp32 kernels' grad_x on the widened inputs rounded once; the other gradients are fp32 and bit-identical to
    theirs."""
    # grad_y: a map like x (16-bit x: or an fp32 one); with up_shape, the forward's `up` requirement on W
    if not (_map_ok(x, weight, bias, groups) and _map_ok(grad_y, weight, bias, groups) and grad_y.shape == x.shape
            and (grad_y.dtype == x.dtype or grad_y.dtype == torch.float32)
            and (up_shape is None or x.size(3) % 4 == 0)):
        raise RuntimeError("group_norm_backward needs contiguous NCHW fp32 CUDA grad_y and x of the same shape with H*W "
                           "(and, with up_shape, W) a multiple of 4, and contiguous fp32 [C] weight and bias")
    _check_channel_bias(channel_bias, x)
    _check_mean_rstd(mean_rstd, x, groups)
    N, C, H, W = x.shape
    gx = torch.empty_like(x)
    gw, gb = torch.empty_like(weight), torch.empty_like(bias)
    gcb = torch.empty_like(bias) if with_channel_bias else None
    gup = (torch.empty(N, C, int(up_shape[0]), int(up_shape[1]), dtype=torch.float32, device=x.device) if up_shape
           else None)
    with torch.cuda.device(x.device):
        ws = _workspace(_lib.lib.msda_b200_group_norm_backward_workspace_bytes(N, C), x)
        if x.dtype == torch.float32:
            entry, grads = _lib.lib.msda_b200_group_norm_backward_nchw_f32, (grad_y.data_ptr(),)
        else:                      # exactly one of grad_y (fp32) and grad_y16
            entry = _GN_MIXED[x.dtype]["group_norm_backward_nchw_mixed"]
            grads = (grad_y.data_ptr(), None) if grad_y.dtype == torch.float32 else (None, grad_y.data_ptr())
        rc = entry(
            *grads, x.data_ptr(), _ptr(channel_bias), weight.data_ptr(), bias.data_ptr(),
            mean_rstd.data_ptr(), gx.data_ptr(), gw.data_ptr(), gb.data_ptr(), _ptr(gcb), _ptr(gup), N, C, H, W,
            groups, int(bool(relu)), gup.size(2) if gup is not None else 0, gup.size(3) if gup is not None else 0,
            ws.data_ptr(), torch.cuda.current_stream(x.device).cuda_stream)
    _lib.check(rc, "group_norm_backward")
    return gx, gw, gb, gcb, gup


def group_norm_rows_backward(grad_rows, x, weight, bias, mean_rstd, groups, relu=False, channel_bias=None,
                             with_channel_bias=False):
    """Gradients of ``group_norm_rows_train``: ``(grad_x, grad_weight, grad_bias, grad_channel_bias)`` with ``grad_rows``
    an fp32 [N, H*W, C] view in the rows layout (e.g. the level's slice of the concatenated gradient) and grad_x NCHW
    of x's type (bf16 / fp16 x: the fp32 kernels' grad_x rounded once).  Three launches; deterministic."""
    if not (_map_ok(x, weight, bias, groups) and _rows_view_ok(grad_rows, x)):
        raise RuntimeError("group_norm_rows_backward needs what group_norm_backward needs, channels % 32 == 0 and an "
                           "fp32 [N, H*W, C] grad_rows view with unit channel stride on the same device")
    _check_channel_bias(channel_bias, x)
    _check_mean_rstd(mean_rstd, x, groups)
    N, C, H, W = x.shape
    gx = torch.empty_like(x)
    gw, gb = torch.empty_like(weight), torch.empty_like(bias)
    gcb = torch.empty_like(bias) if with_channel_bias else None
    with torch.cuda.device(x.device):
        ws = _workspace(_lib.lib.msda_b200_group_norm_backward_workspace_bytes(N, C), x)
        entry = (_lib.lib.msda_b200_group_norm_rows_backward_f32 if x.dtype == torch.float32
                 else _GN_MIXED[x.dtype]["group_norm_rows_backward_mixed"])
        rc = entry(
            grad_rows.data_ptr(), grad_rows.stride(1), grad_rows.stride(0), x.data_ptr(), _ptr(channel_bias),
            weight.data_ptr(), bias.data_ptr(), mean_rstd.data_ptr(), gx.data_ptr(), gw.data_ptr(), gb.data_ptr(),
            _ptr(gcb), N, C, H * W, groups, int(bool(relu)), ws.data_ptr(), torch.cuda.current_stream(x.device).cuda_stream)
    _lib.check(rc, "group_norm_rows_backward")
    return gx, gw, gb, gcb
