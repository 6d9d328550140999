"""Autograd wrapper with the reference's interface:
``MSDeformAttnFunction.apply(value, spatial_shapes, level_start_index, sampling_locations,
attention_weights, im2col_step)`` (ops/functions/ms_deform_attn_func.py:35-52).

The reference's own ``MSDeformAttnFunction`` also runs unchanged on top of
``dropin/MultiScaleDeformableAttention.py``; this mirror exists so that code on a box
without the reference checkout (the GPU box, bench.py) has the same entry point.
"""
from __future__ import annotations

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import ops


class MSDeformAttnFunction(Function):
    @staticmethod
    def forward(ctx, value, value_spatial_shapes, value_level_start_index, sampling_locations,
                attention_weights, im2col_step):
        ctx.im2col_step = im2col_step
        output = ops.ms_deform_attn_forward(value, value_spatial_shapes, value_level_start_index,
                                            sampling_locations, attention_weights, im2col_step)
        ctx.save_for_backward(value, value_spatial_shapes, value_level_start_index,
                              sampling_locations, attention_weights)
        return output

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        value, shapes, lsi, loc, w = ctx.saved_tensors
        grad_value, grad_loc, grad_w = ops.ms_deform_attn_backward(
            value, shapes, lsi, loc, w, grad_output, ctx.im2col_step)
        return grad_value, None, None, grad_loc, grad_w, None


class MSDeformAttnMixedFunction(Function):
    """``MSDeformAttnFunction`` for mixed precision (torch.autocast): same ``apply`` signature, a bf16 / fp16
    ``value`` (output and grad_value in its dtype) with fp32 ``sampling_locations`` / ``attention_weights`` (and
    fp32 gradients for them); every sum in fp32 (ops.ms_deform_attn_mixed_forward / _backward)."""

    @staticmethod
    def forward(ctx, value, value_spatial_shapes, value_level_start_index, sampling_locations,
                attention_weights, im2col_step):
        ctx.im2col_step = im2col_step
        output = ops.ms_deform_attn_mixed_forward(value, value_spatial_shapes, value_level_start_index,
                                                  sampling_locations, attention_weights, im2col_step)
        ctx.save_for_backward(value, value_spatial_shapes, value_level_start_index,
                              sampling_locations, attention_weights)
        return output

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        value, shapes, lsi, loc, w = ctx.saved_tensors
        grad_value, grad_loc, grad_w = ops.ms_deform_attn_mixed_backward(
            value, shapes, lsi, loc, w, grad_output.contiguous(), ctx.im2col_step)
        return grad_value, None, None, grad_loc, grad_w, None


class MSDeformAttnFusedFunction(Function):
    """``apply(value, spatial_shapes, level_start_index, reference_points, sampling_offsets,
    attn_logits)`` -- the op with its caller's softmax and location arithmetic
    (ops/modules/ms_deform_attn.py:105-112) inside the kernels.  Gradients flow to value,
    sampling_offsets and attn_logits; reference_points are treated as constants (they are in the
    encoder, msdeformattn.py:152-166)."""

    @staticmethod
    def forward(ctx, value, spatial_shapes, level_start_index, reference_points, sampling_offsets,
                attn_logits):
        output = ops.ms_deform_attn_fused_forward(value, spatial_shapes, level_start_index,
                                                  reference_points, sampling_offsets, attn_logits)
        ctx.save_for_backward(value, spatial_shapes, level_start_index, reference_points,
                              sampling_offsets, attn_logits)
        return output

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        value, shapes, lsi, ref, off, logits = ctx.saved_tensors
        grad_value, grad_off, grad_logits = ops.ms_deform_attn_fused_backward(
            value, shapes, lsi, ref, off, logits, grad_output)
        return grad_value, None, None, None, grad_off, grad_logits


class LinearTF32x3Function(Function):
    """``apply(x, weight, bias)`` = ``F.linear`` with all three GEMMs on the tensor cores: forward and
    input gradient (``grad_y @ weight``) through ops.linear_tf32x3, weight and bias gradient
    (``grad_y^T @ x``, column sums of ``grad_y``) through ops.linear_wgrad, which reduces over the rows
    without transposing the operands in memory (0.15 ms against 0.53 + 0.12 ms for torch's fp32 GEMM and
    column sum at 172 032 x 256 x 256).  Needs in_features and out_features divisible by 32.
    ``apply(x, weight, bias, True)`` = ``F.relu(F.linear(...))`` with the ReLU in the GEMM's epilogue (no separate
    pass over the output); its backward masks ``grad_y`` where the saved output is zero, as ``F.relu`` does.
    ``apply(x, weight, bias, True, p)`` = ``F.dropout(F.relu(F.linear(...)), p, training=True)`` (the FFN's hidden
    activation, msdeformattn.py:126-130): the mask is drawn by torch's own dropout kernel (same generator stream
    as ``F.dropout``); a kept element is positive exactly where the ReLU was active, so the backward needs ONE pass
    over the hidden gradient (``threshold_backward`` against the saved output) instead of two, and the 1/(1-p)
    scale moves onto the small tensors (the transposed weight, grad_weight, grad_bias)."""

    @staticmethod
    def supported(x, weight) -> bool:
        return (ops.linear_tf32x3_supported(x, weight) and x.is_contiguous()
                and weight.size(0) % 32 == 0 and weight.size(1) % 32 == 0)

    @staticmethod
    def forward(ctx, x, weight, bias, relu=False, dropout_p=0.0):
        if dropout_p and not (relu and 0.0 < dropout_p < 1.0):
            raise ValueError("dropout_p needs relu=True and 0 < p < 1")
        y = ops.linear_tf32x3(x, weight.contiguous(), bias, relu=relu)
        ctx.has_bias = bias is not None
        ctx.relu = bool(relu)
        ctx.scale = 1.0
        if dropout_p:
            y, _ = torch.native_dropout(y, float(dropout_p), True)       # y * mask / (1 - p)
            ctx.scale = 1.0 / (1.0 - float(dropout_p))
        if relu:
            ctx.save_for_backward(x, weight, y)
        else:
            ctx.save_for_backward(x, weight)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_y):
        if ctx.relu:
            x, weight, y = ctx.saved_tensors
            # F.relu's backward; with dropout, y > 0 exactly where the element was kept AND the ReLU was active,
            # and the scale 1/(1-p) is applied to the results below instead of to this (large) tensor
            grad_y = torch.ops.aten.threshold_backward(grad_y, y, 0)
        else:
            x, weight = ctx.saved_tensors
        grad_y = grad_y.contiguous()
        scale = ctx.scale
        grad_x = grad_w = grad_b = None
        if ctx.needs_input_grad[0]:
            wt = weight.t().contiguous() if scale == 1.0 else (weight.t() * scale).contiguous()
            grad_x = ops.linear_tf32x3(grad_y, wt, None)
        g2 = grad_y.reshape(-1, grad_y.size(-1))
        want_b = ctx.has_bias and ctx.needs_input_grad[2]
        if ctx.needs_input_grad[1]:
            x2 = x.reshape(-1, x.size(-1))
            if ops.linear_wgrad_supported(g2, x2):
                grad_w, grad_b = ops.linear_wgrad(g2, x2, with_bias=want_b)
            else:
                grad_w = g2.t() @ x2
        if want_b and grad_b is None:
            grad_b = g2.sum(0)
        if scale != 1.0:
            grad_w = grad_w * scale if grad_w is not None else None
            grad_b = grad_b * scale if grad_b is not None else None
        return grad_x, grad_w, grad_b, None, None


class LinearMixedFunction(Function):
    """``apply(x16, weight, bias, relu=False, dropout_p=0.0)``: ``LinearTF32x3Function`` under torch.autocast.  ``x16``
    is bf16 / fp16, ``weight`` and ``bias`` (may be None) the fp32 parameters; the weight is cast to x16's dtype once
    per call.  = ``F.linear(x16, weight, bias)`` as autocast computes it (bias added to the fp32 accumulator, one
    rounding; ops.linear_mixed), with ``relu`` in the GEMM's epilogue and ``dropout_p`` drawn by torch's own dropout
    kernel on the 16-bit output.  Backward: one ``threshold_backward`` when ``relu`` is set, the input gradient (in x16's
    dtype) as torch's 16-bit GEMM -- faster than the library kernel at every measured shape (ops.linear_mixed_preferred)
    -- or, with torch.use_deterministic_algorithms(True), on the library kernel, and the fp32 weight and bias gradients
    of ops.linear_mixed_wgrad, which go to the fp32 parameters without a 16-bit rounding; the 1/(1-p) scale is applied
    to the transposed weight and to those."""

    @staticmethod
    def supported(x16, weight, bias=None) -> bool:
        """Whether the kernels cover ``x16`` with the fp32 parameters ``weight`` [out, in] and ``bias``."""
        return (isinstance(weight, torch.Tensor) and weight.dtype == torch.float32 and weight.dim() == 2
                and weight.is_contiguous()
                and ops.linear_mixed_shapes_supported(x16, weight.size(0), weight.size(1), bias)
                and weight.device == x16.device)

    @staticmethod
    def forward(ctx, x16, weight, bias, relu=False, dropout_p=0.0):
        if dropout_p and not (relu and 0.0 < dropout_p < 1.0):
            raise ValueError("dropout_p needs relu=True and 0 < p < 1")
        w16 = weight.detach().to(x16.dtype)
        y = ops.linear_mixed(x16, w16, bias, relu=relu)
        ctx.has_bias = bias is not None
        ctx.relu = bool(relu)
        ctx.scale = 1.0
        if dropout_p:
            y, _ = torch.native_dropout(y, float(dropout_p), True)       # y * mask / (1 - p)
            ctx.scale = 1.0 / (1.0 - float(dropout_p))
        ctx.save_for_backward(x16, w16, y if relu else None, weight if dropout_p else None)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_y):
        x16, w16, y, weight = ctx.saved_tensors
        grad_y = grad_y.to(x16.dtype)
        if ctx.relu:
            # F.relu's backward; with dropout, y > 0 exactly where the element was kept AND the ReLU was active
            grad_y = torch.ops.aten.threshold_backward(grad_y, y, 0)
        g2 = _aligned(grad_y.reshape(-1, grad_y.size(-1)))
        scale = ctx.scale
        grad_x = grad_w = grad_b = None
        if ctx.needs_input_grad[0]:
            w_in = w16 if scale == 1.0 else (weight * scale).to(x16.dtype)          # [out, in]
            if ops._deterministic() or ops.linear_mixed_preferred(g2.size(0), w_in.size(1), w_in.size(0), False,
                                                                   "input_gradient"):
                grad_x = ops.linear_mixed(g2, w_in.t().contiguous()).view(x16.shape)
            else:
                grad_x = (g2 @ w_in).view(x16.shape)
        want_b = ctx.has_bias and ctx.needs_input_grad[2]
        if ctx.needs_input_grad[1] or want_b:
            grad_w, grad_b = ops.linear_mixed_wgrad(g2, x16.reshape(-1, x16.size(-1)), with_bias=want_b)
            if not ctx.needs_input_grad[1]:
                grad_w = None
        if scale != 1.0:
            grad_w = grad_w * scale if grad_w is not None else None
            grad_b = grad_b * scale if grad_b is not None else None
        return grad_x, grad_w, grad_b, None, None


class AddLayerNormFunction(Function):
    """``apply(x, residual, weight, bias, eps)`` = ``F.layer_norm(x + residual, (C,), weight, bias, eps)`` with one
    fused kernel each way (ops.add_layernorm / add_layernorm_backward); C in {128, 256}."""

    @staticmethod
    def supported(x, residual, weight) -> bool:
        return ops.add_layernorm_supported(x, residual, weight) and x.size(-1) in (128, 256) and residual is not None

    @staticmethod
    def forward(ctx, x, residual, weight, bias, eps):
        ctx.save_for_backward(x, residual, weight)
        ctx.eps = eps
        return ops.add_layernorm(x, residual, weight, bias, eps)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_y):
        x, residual, weight = ctx.saved_tensors
        gv, gg, gb = ops.add_layernorm_backward(grad_y.contiguous(), x, residual, weight, ctx.eps)
        return gv, gv, gg, gb, None


class AddLayerNormMixedFunction(Function):
    """``apply(x, residual16, weight, bias, eps)`` -> ``(y, y16)`` with ``y = F.layer_norm(x + residual16.float(), (C,),
    weight, bias, eps)`` (fp32: the residual stream under torch.autocast) and ``y16 = y.to(residual16.dtype)`` (the copy
    the next GEMMs read) -- one kernel each way (ops.add_layernorm_mixed / add_layernorm_mixed_backward); C in {128,
    256}.  Either output may go unused: its gradient is then absent, and the backward adds the two gradients in fp32
    where both are present, as autograd does for torch's composition.  Returns an fp32 grad_x and a grad_residual of
    residual16's dtype."""

    @staticmethod
    def supported(x, residual, weight) -> bool:
        return ops.add_layernorm_mixed_backward_supported(x, residual, weight)

    @staticmethod
    def forward(ctx, x, residual, weight, bias, eps):
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(x, residual, weight)
        ctx.eps = eps
        return ops.add_layernorm_mixed(x, residual, weight, bias, eps)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_y, grad_y16):
        if grad_y is None and grad_y16 is None:
            return None, None, None, None, None
        x, residual, weight = ctx.saved_tensors
        gx, gr, gg, gb = ops.add_layernorm_mixed_backward(
            _aligned(grad_y) if grad_y is not None else None,
            _aligned(grad_y16) if grad_y16 is not None else None, x, residual, weight, ctx.eps)
        return gx, gr, gg, gb, None


def _aligned(t):
    """`t` contiguous and 16-byte aligned (the kernels' 128-bit accesses); copies only when it is not."""
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


class GroupNormFunction(Function):
    """``apply(x, weight, bias, channel_bias, up, groups, eps, relu)`` =
    ``F.group_norm(x + channel_bias[None, :, None, None], groups, weight, bias, eps)`` [-> ``F.relu``]
    [+ ``F.interpolate(up, size=x.shape[-2:], mode="bilinear", align_corners=False)``] -- the pixel decoder's
    GroupNorm epilogues (msdeformattn.py:233-248, :369-379) -- with the fused kernels both ways: two launches forward
    (ops.group_norm_train, bit-identical to ops.group_norm), three backward, four with the gradient of ``up``
    (ops.group_norm_backward).  ``channel_bias`` and ``up`` may be None.  Saves x and the [N, groups, 2] statistics,
    not the output; the ReLU mask is rebuilt from x with the forward's own arithmetic.

    A bf16 / fp16 ``x`` (torch.autocast) is saved as it is, not widened; the result is fp32 (``out_dtype`` None, what
    autocast's ``F.group_norm`` returns) or its copy rounded to x's type (``out_dtype=x.dtype``), and grad_x has x's
    type."""

    @staticmethod
    def forward(ctx, x, weight, bias, channel_bias, up, groups, eps, relu, out_dtype=None):
        y, mean_rstd = ops.group_norm_train(x, weight, bias, groups, eps, relu=relu, up=up, channel_bias=channel_bias,
                                            out_dtype=out_dtype)
        ctx.save_for_backward(x, weight, bias, channel_bias, mean_rstd)
        ctx.groups, ctx.relu = groups, bool(relu)
        ctx.up_shape = tuple(up.shape[-2:]) if up is not None else None
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_y):
        x, weight, bias, channel_bias, mean_rstd = ctx.saved_tensors
        need = ctx.needs_input_grad
        gx, gw, gb, gcb, gup = ops.group_norm_backward(
            _aligned(grad_y), x, weight, bias, mean_rstd, ctx.groups, relu=ctx.relu, channel_bias=channel_bias,
            up_shape=ctx.up_shape if need[4] else None, with_channel_bias=channel_bias is not None and need[3])
        return (gx if need[0] else None, gw if need[1] else None, gb if need[2] else None, gcb, gup, None, None, None,
                None)


class GroupNormRowsFunction(Function):
    """``apply(groups, eps, x_0, weight_0, bias_0, channel_bias_0, x_1, ...)`` = the encoder input
    ``torch.cat([F.group_norm(x_i + channel_bias_i, groups, weight_i, bias_i, eps).flatten(2).transpose(1, 2)], 1)``
    ([N, sum of H_i * W_i, C]) of the pixel decoder's input projections (msdeformattn.py:341-345, :72-79) as ONE
    autograd node: every level's GroupNorm writes its rows of the concatenated tensor (ops.group_norm_rows_train) and
    its backward reads them back from the concatenated gradient (ops.group_norm_rows_backward), so neither the
    transposing ``cat`` nor its backward runs.  ``channel_bias_i`` may be None.  Two launches per level forward,
    three backward.  The levels may be bf16 / fp16 (torch.autocast), all of one type: the output stays fp32 and each
    grad_x has its level's type."""

    @staticmethod
    def forward(ctx, groups, eps, *level_args):
        levels = [level_args[i:i + 4] for i in range(0, len(level_args), 4)]
        x0 = levels[0][0]
        if any(x.dtype != x0.dtype for x, _, _, _ in levels):
            raise RuntimeError("GroupNormRowsFunction: all levels must have one dtype")
        sizes = [x.size(2) * x.size(3) for x, _, _, _ in levels]
        out = x0.new_empty((x0.size(0), sum(sizes), x0.size(1)), dtype=torch.float32)
        saved, start = [], 0
        for (x, weight, bias, channel_bias), hw in zip(levels, sizes):
            mean_rstd = ops.group_norm_rows_train(x, weight, bias, groups, eps, out[:, start:start + hw],
                                                  channel_bias=channel_bias)
            saved += [x, weight, bias, channel_bias, mean_rstd]
            start += hw
        ctx.save_for_backward(*saved)
        ctx.groups, ctx.sizes = groups, sizes
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        grad_out = _aligned(grad_out)
        saved, need = ctx.saved_tensors, ctx.needs_input_grad
        grads, start = [None, None], 0
        for i, hw in enumerate(ctx.sizes):
            x, weight, bias, channel_bias, mean_rstd = saved[5 * i:5 * i + 5]
            gx, gw, gb, gcb = ops.group_norm_rows_backward(
                grad_out[:, start:start + hw], x, weight, bias, mean_rstd, ctx.groups, channel_bias=channel_bias,
                with_channel_bias=channel_bias is not None and need[2 + 4 * i + 3])
            k = 2 + 4 * i
            grads += [gx if need[k] else None, gw if need[k + 1] else None, gb if need[k + 2] else None, gcb]
            start += hw
        return tuple(grads)
