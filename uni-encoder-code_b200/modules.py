"""Host-side mirror of the callers on either side of the MSDA op, for boxes that do not have
the reference checkout (the GPU box, bench tools) and for the "next" rows of SURVEY.md section 8f.

Same class names, constructor arguments, parameter names (so reference checkpoints load with
``load_state_dict``) and forward signatures as the reference:

* ``MSDeformAttn``                         ops/modules/ms_deform_attn.py:35-126
* ``MSDeformAttnTransformerEncoderLayer``  model/modeling/pixel_decoder/msdeformattn.py:102-142
* ``MSDeformAttnTransformerEncoder``       msdeformattn.py:145-176
* ``MSDeformAttnTransformerEncoderOnly``   msdeformattn.py:26-99

The reference's own classes also run unchanged on the drop-in shim; these mirrors exist so the
encoder-level configs (BASELINE configs[2..4]) can be measured without it, and differ only where
SURVEY 8f ranks a saving: reference points are built without iterating a CUDA tensor on the host
(msdeformattn.py:154 syncs), and the encoder does not allocate / apply the all-False padding masks
(msdeformattn.py:68-69, ms_deform_attn.py:102-103 rewrite ``value`` with an unchanged copy).

The core op is always the CUDA one (``MSDeformAttnFunction``); there is no CPU branch.  Tests of the
host logic on CPU pass ``core=`` explicitly.
"""
from __future__ import annotations

import copy
import math
import weakref
from typing import Callable, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F
from torch import nn

from . import ops
from .functions import (AddLayerNormFunction, AddLayerNormMixedFunction, LinearMixedFunction, LinearTF32x3Function,
                        MSDeformAttnFunction, MSDeformAttnFusedFunction, MSDeformAttnMixedFunction)

CoreFn = Callable[..., torch.Tensor]


class ShapeCache:
    """Small LRU for shape-keyed device constants (position embeddings, reference points, level
    tensors).  The reference recomputes these on every forward and holds nothing; caching them is
    what makes the decoder CUDA-graph capturable, but datasets with variable resolution (ADE20K,
    COCO) present thousands of distinct pyramids, so only the most recent `maxsize` shapes stay
    resident -- a deployment that captures graphs uses a fixed set of shapes well below that."""

    def __init__(self, maxsize: int = 8):
        from collections import OrderedDict
        self.maxsize, self._d = maxsize, OrderedDict()

    def get(self, key):
        hit = self._d.get(key)
        if hit is not None:
            self._d.move_to_end(key)
        return hit

    def put(self, key, value):
        self._d[key] = value
        self._d.move_to_end(key)
        while len(self._d) > self.maxsize:
            self._d.popitem(last=False)
        return value

    def __len__(self):
        return len(self._d)

    def __contains__(self, key):
        return key in self._d

    def clear(self):
        self._d.clear()


def _version_of(t: torch.Tensor) -> int:
    """In-place modification counter for cache keys; inference tensors (created under
    torch.inference_mode()) do not track one -- reading ._version on them raises."""
    return -1 if t.is_inference() else t._version


def _capturing(t: torch.Tensor) -> bool:
    """True while a CUDA graph is being captured on the current stream: results computed now are not materialised
    until the graph is replayed, so nothing computed during capture may be kept in a cache that eager calls read."""
    return t.is_cuda and torch.cuda.is_current_stream_capturing()


def _presplit_of(layer: nn.Linear):
    """The split form of `layer.weight` for the inference GEMM, computed once per weight version (the weight does
    not change between inference calls; an in-place update or a new tensor rebuilds it)."""
    w = layer.weight
    key = (w.data_ptr(), _version_of(w), tuple(w.shape), str(w.device))
    hit = layer.__dict__.get("_tf32x3_presplit")
    if hit is None or hit[0] != key:
        hit = (key, ops.split_weight(w))
        if not _capturing(w):
            layer.__dict__["_tf32x3_presplit"] = hit
    return hit[1]


def _weight16_of(w: torch.Tensor, owner: dict, dtype):
    """`w` cast to `dtype` for the inference GEMM under autocast, kept in `owner` (a module's __dict__) per weight
    version and per weight tensor (a new tensor at the old address with an equal version is not served the old copy);
    not kept while a CUDA graph is captured."""
    key = (w.data_ptr(), _version_of(w), tuple(w.shape), str(w.device), dtype)
    hit = owner.get("_weight16")
    if hit is None or hit[0] != key or hit[1]() is not w:
        hit = (key, weakref.ref(w), w.detach().to(dtype))
        if not _capturing(w):
            owner["_weight16"] = hit
    return hit[2]


def _autocast_dtype():
    """The 16-bit type of the active CUDA torch.autocast, or None (no context, a disabled one, or another type)."""
    if not torch.is_autocast_enabled("cuda"):
        return None
    dtype = torch.get_autocast_dtype("cuda")
    return dtype if dtype in (torch.bfloat16, torch.float16) else None


def _resolve(impl: str) -> str:
    """linear="autocast" is linear="tf32x3" unless a bf16 / fp16 CUDA autocast is active; then it stays "autocast":
    torch's autocast GEMMs and the mixed-precision residual + LayerNorm kernels (`_add_norm_mixed`)."""
    if impl == "autocast" and _autocast_dtype() is None:
        return "tf32x3"
    return impl


def _linear(layer: nn.Linear, x, impl: str, relu: bool = False):
    """``layer(x)`` (+ ReLU).  impl == "tf32x3" selects the inference kernels of SURVEY 8f.3 (this GEMM and the
    fused residual + LayerNorm of `_add_norm`): in inference (autograd off) the fp32 GEMM runs on the
    tensor cores as an error-compensated 3xTF32 product (ops.linear_tf32x3, SURVEY 8f.3); with autograd
    on, the forward and the input-gradient GEMMs do (LinearTF32x3Function; the weight gradient stays a
    torch GEMM); for any shape the kernel does not cover torch's own fp32 GEMM is used as in the reference.
    impl == "autocast": see `_resolve`; under a 16-bit autocast the 16-bit GEMM of `_linear_mixed`, or torch's
    autocast GEMM for shapes it does not cover."""
    impl = _resolve(impl)
    if impl == "autocast":
        y = _linear_mixed(layer, x, relu)
        if y is not None:
            return y
    if impl == "tf32x3" and not torch.is_grad_enabled() and x.is_contiguous() \
            and ops.linear_tf32x3_supported(x, layer.weight):
        return ops.linear_tf32x3(x, layer.weight, layer.bias, relu=relu, presplit=_presplit_of(layer))
    if impl == "tf32x3" and torch.is_grad_enabled() and LinearTF32x3Function.supported(x, layer.weight):
        # all three GEMMs on the tensor cores; the ReLU rides in the forward GEMM's epilogue
        return LinearTF32x3Function.apply(x, layer.weight, layer.bias, relu)
    if impl not in ("torch", "tf32x3", "autocast"):
        raise ValueError(f"unknown linear implementation {impl!r}")
    y = layer(x)
    return F.relu(y) if relu else y


def _to_autocast16(x):
    """`x` as the active autocast's 16-bit type: an fp32 tensor is cast (once, for every GEMM that reads it)."""
    dtype = _autocast_dtype()
    return x.to(dtype) if dtype is not None and x.dtype == torch.float32 else x


def _linear_mixed(layer: nn.Linear, x, relu: bool = False, dropout_p: float = 0.0):
    """Under a 16-bit autocast: ``layer(x)`` (+ ReLU, + dropout: autograd only) on the library's 16-bit GEMM with
    the fp32 bias in its epilogue -- ops.linear_mixed with the 16-bit weight cached per version in inference,
    LinearMixedFunction (fp32 weight and bias gradients) with autograd -- or None where it does not apply."""
    dtype = _autocast_dtype()
    w, b = layer.weight, layer.bias
    if dtype is None or w.dtype != torch.float32 or (b is not None and b.dtype != torch.float32):
        return None
    x16 = _to_autocast16(x)
    if x16.dtype != dtype or not LinearMixedFunction.supported(x16, w, b):
        return None
    if torch.is_grad_enabled():
        # the whole node (forward, input and weight gradients) is faster than torch's at every measured site
        return LinearMixedFunction.apply(x16, w, b, relu, dropout_p)
    if not ops.linear_mixed_preferred(x16.numel() // x16.size(-1), w.size(0), w.size(1), relu, "forward"):
        return None                         # measured slower than torch's GEMM at this shape
    return ops.linear_mixed(x16, _weight16_of(w, layer.__dict__, dtype), b, relu=relu)


def _add_norm(norm: nn.LayerNorm, x, sublayer_out, impl: str):
    """``norm(x + sublayer_out)``; impl == "tf32x3" (inference): one fused pass (ops.add_layernorm)."""
    impl = _resolve(impl)
    if impl == "tf32x3" and not torch.is_grad_enabled() and norm.elementwise_affine \
            and ops.add_layernorm_supported(x, sublayer_out, norm.weight, norm.bias, need_bias=True):
        return ops.add_layernorm(x, sublayer_out, norm.weight, norm.bias, norm.eps)
    if impl == "tf32x3" and torch.is_grad_enabled() and norm.elementwise_affine \
            and norm.bias is not None and sublayer_out.is_contiguous() \
            and AddLayerNormFunction.supported(x, sublayer_out, norm.weight):
        return AddLayerNormFunction.apply(x, sublayer_out, norm.weight, norm.bias, norm.eps)
    return norm(x + sublayer_out)


def _add_norm_mixed(norm: nn.LayerNorm, x, sublayer_out):
    """Under a 16-bit autocast: (``norm(x + sublayer_out)``, its 16-bit copy for the next GEMMs or None).  An fp32
    residual stream ``x`` and a 16-bit ``sublayer_out`` go through the mixed-precision kernels (ops.add_layernorm_mixed
    without autograd, AddLayerNormMixedFunction with it), which also write the copy autocast's own cast would give;
    whatever they do not cover takes torch's composition (no copy: the GEMMs cast)."""
    if norm.elementwise_affine and norm.bias is not None and sublayer_out.dtype == _autocast_dtype():
        if not torch.is_grad_enabled() \
                and ops.add_layernorm_mixed_supported(x, sublayer_out, norm.weight, norm.bias, need_bias=True):
            return ops.add_layernorm_mixed(x, sublayer_out, norm.weight, norm.bias, norm.eps)
        if torch.is_grad_enabled() and AddLayerNormMixedFunction.supported(x, sublayer_out, norm.weight) \
                and ops.add_layernorm_mixed_supported(x, sublayer_out, norm.weight, norm.bias, need_bias=True):
            return AddLayerNormMixedFunction.apply(x, sublayer_out, norm.weight, norm.bias, norm.eps)
    return norm(x + sublayer_out), None


def _cuda_core(value, spatial_shapes, level_start_index, sampling_locations, attention_weights,
               im2col_step):
    if value.dtype in (torch.bfloat16, torch.float16):
        # mixed precision (autocast): 16-bit value rows, locations and weights in fp32 (upcasting them is exact)
        return MSDeformAttnMixedFunction.apply(value, spatial_shapes, level_start_index, sampling_locations.float(),
                                               attention_weights.float(), im2col_step)
    return MSDeformAttnFunction.apply(value, spatial_shapes, level_start_index, sampling_locations,
                                      attention_weights, im2col_step)


class MSDeformAttn(nn.Module):
    """Multi-scale deformable attention module (ms_deform_attn.py:35-126)."""

    def __init__(self, d_model=256, n_levels=4, n_heads=8, n_points=4, core: Optional[CoreFn] = None,
                 fused: bool = False, linear: str = "torch"):
        """`fused=True` (not in the reference): softmax and location arithmetic run inside the
        kernels whenever the shapes allow (SURVEY 8f.1); results agree to rounding.
        `linear="tf32x3"` (not in the reference): see `_linear`; `linear="autocast"`: see `_resolve`."""
        super().__init__()
        self.fused = fused
        self.linear = linear
        if d_model % n_heads:
            raise ValueError(f"d_model must be divisible by n_heads, but got {d_model} and {n_heads}")
        self.im2col_step = 128                    # ms_deform_attn.py:55
        self.d_model, self.n_levels, self.n_heads, self.n_points = d_model, n_levels, n_heads, n_points
        self.sampling_offsets = nn.Linear(d_model, n_heads * n_levels * n_points * 2)
        self.attention_weights = nn.Linear(d_model, n_heads * n_levels * n_points)
        self.value_proj = nn.Linear(d_model, d_model)
        self.output_proj = nn.Linear(d_model, d_model)
        self._core = core or _cuda_core
        self._reset_parameters()

    def _reset_parameters(self):
        # ms_deform_attn.py:69-83: zero offset weights, offsets biased along 8 compass directions
        # scaled by the point index; uniform attention; xavier value / output projections
        with torch.no_grad():
            self.sampling_offsets.weight.zero_()
            ang = torch.arange(self.n_heads, dtype=torch.float32) * (2.0 * math.pi / self.n_heads)
            dirs = torch.stack((ang.cos(), ang.sin()), -1)
            dirs = dirs / dirs.abs().amax(-1, keepdim=True)
            scale = torch.arange(1, self.n_points + 1, dtype=torch.float32).view(1, 1, -1, 1)
            bias = dirs.view(self.n_heads, 1, 1, 2) * scale            # broadcast over levels
            bias = bias.expand(self.n_heads, self.n_levels, self.n_points, 2)
            self.sampling_offsets.bias.copy_(bias.reshape(-1))
            self.attention_weights.weight.zero_()
            self.attention_weights.bias.zero_()
            nn.init.xavier_uniform_(self.value_proj.weight)
            self.value_proj.bias.zero_()
            nn.init.xavier_uniform_(self.output_proj.weight)
            self.output_proj.bias.zero_()

    def sampling_inputs(self, query, reference_points, input_spatial_shapes):
        """(sampling_locations [N,Lq,M,L,P,2], attention_weights [N,Lq,M,L,P]) from the query
        (ms_deform_attn.py:105-118)."""
        N, Lq, _ = query.shape
        M, L, P = self.n_heads, self.n_levels, self.n_points
        offsets = _linear(self.sampling_offsets, query, self.linear).view(N, Lq, M, L, P, 2)
        weights = F.softmax(_linear(self.attention_weights, query, self.linear).view(N, Lq, M, L * P), -1).view(N, Lq, M, L, P)
        if offsets.dtype in (torch.bfloat16, torch.float16):
            offsets = offsets.float()       # autocast: the locations are formed in fp32 (a 16-bit one is off by up to
            #                                 half a pixel at W = 256)
        if reference_points.shape[-1] == 2:
            wh = input_spatial_shapes.flip(-1).to(offsets.dtype)       # (W_l, H_l)
            loc = reference_points[:, :, None, :, None, :] + offsets / wh[None, None, None, :, None, :]
        elif reference_points.shape[-1] == 4:
            loc = (reference_points[:, :, None, :, None, :2]
                   + offsets / P * reference_points[:, :, None, :, None, 2:] * 0.5)
        else:
            raise ValueError(
                f"Last dim of reference_points must be 2 or 4, but get {reference_points.shape[-1]} instead.")
        return loc, weights

    def project_value(self, input_flatten, input_padding_mask=None):
        N, S, _ = input_flatten.shape
        value = _linear(self.value_proj, input_flatten, self.linear)
        if input_padding_mask is not None:
            value = value.masked_fill(input_padding_mask[..., None], 0.0)
        return value.view(N, S, self.n_heads, self.d_model // self.n_heads)

    def forward(self, query, reference_points, input_flatten, input_spatial_shapes,
                input_level_start_index, input_padding_mask=None):
        value = self.project_value(input_flatten, input_padding_mask)
        if _resolve(self.linear) == "autocast":
            query = _to_autocast16(query)      # read by two GEMMs: cast once
        # fp32, or under autocast a 16-bit value whose offsets / logits come out in the same type (fused_supported)
        if self.fused and self._core is _cuda_core and not reference_points.requires_grad \
                and value.dtype in (torch.float32, torch.bfloat16, torch.float16):
            N, Lq, _ = query.shape
            offsets = _linear(self.sampling_offsets, query, self.linear).view(
                N, Lq, self.n_heads, self.n_levels, self.n_points, 2)
            logits = _linear(self.attention_weights, query, self.linear).view(
                N, Lq, self.n_heads, self.n_levels * self.n_points)
            ref = reference_points
            if ref.dim() == 4 and ref.stride(0) == 0:        # expanded over the batch: pass one copy
                ref = ref[:1]
            ref = ref.contiguous()
            if ops.fused_supported(value, ref, offsets, logits):
                out = MSDeformAttnFusedFunction.apply(value, input_spatial_shapes, input_level_start_index,
                                                      ref, offsets, logits)
                return _linear(self.output_proj, out, self.linear)
        loc, weights = self.sampling_inputs(query, reference_points, input_spatial_shapes)
        out = self._core(value, input_spatial_shapes, input_level_start_index, loc.contiguous(),
                         weights.contiguous(), self.im2col_step)
        return _linear(self.output_proj, out, self.linear)

    # ---- inference with a position embedding shared by the batch (SURVEY 8f.3 / 8f.4) ----
    def can_fold_pos(self, src, pos, reference_points, padding_mask=None) -> bool:
        """Whether `forward_shared_pos` applies: inference kernels on, no mask, 2-d reference points, and
        `pos` [N or 1, S, C] holding the same rows for every image (batch stride 0, as the pixel decoder's
        sine embedding + level embedding is)."""
        if _resolve(self.linear) == "autocast":
            return self._can_fold_pos_mixed(src, pos, reference_points, padding_mask)
        return (self.fused and _resolve(self.linear) == "tf32x3" and self._core is _cuda_core
                and not torch.is_grad_enabled() and padding_mask is None and pos is not None
                and pos.dim() == 3 and (pos.size(0) == 1 or pos.stride(0) == 0)
                and pos.shape[1:] == src.shape[1:] and pos[0].is_contiguous()
                and src.is_cuda and src.dtype == torch.float32 and src.is_contiguous()
                and pos.dtype == torch.float32 and pos.device == src.device
                and reference_points.dim() == 4 and reference_points.size(-1) == 2
                and not reference_points.requires_grad
                and self.d_model // self.n_heads == 32 and self.n_levels * self.n_points in (4, 8, 12, 16)
                and ops.linear_tf32x3_supported(src, self.sampling_offsets.weight)
                and self.sampling_offsets.bias is not None and self.attention_weights.bias is not None)

    def _can_fold_pos_mixed(self, src, pos, reference_points, padding_mask) -> bool:
        """`can_fold_pos` under a 16-bit autocast (linear="autocast"): the same conditions, with the query GEMM run by
        autocast and the fused forward the 16-bit packed one (ops.ms_deform_attn_fused_mixed_forward_packed)."""
        return (self.fused and self._core is _cuda_core and not torch.is_grad_enabled() and padding_mask is None
                and pos is not None and pos.dim() == 3 and (pos.size(0) == 1 or pos.stride(0) == 0)
                and pos.shape[1:] == src.shape[1:] and pos[0].is_contiguous()
                and src.is_cuda and src.dtype == torch.float32 and pos.dtype == torch.float32
                and pos.device == src.device and reference_points.dim() == 4 and reference_points.size(-1) == 2
                and not reference_points.requires_grad
                and self.d_model // self.n_heads == 32 and self.n_levels * self.n_points in (4, 8, 12, 16)
                and ops.linear_tf32x3_supported(pos[0], self.sampling_offsets.weight)
                and self.sampling_offsets.bias is not None and self.attention_weights.bias is not None)

    def _query_projection(self, pos_rows):
        """(stacked weight [3*M*L*P, C] of sampling_offsets and attention_weights, table [S, 3*M*L*P] =
        pos_rows @ weight^T + stacked bias, the stacked weight in split form), rebuilt when a parameter or the
        embedding changes."""
        params = (self.sampling_offsets.weight, self.sampling_offsets.bias,
                  self.attention_weights.weight, self.attention_weights.bias)
        key = tuple((t.data_ptr(), _version_of(t)) for t in params + (pos_rows,)) + (tuple(pos_rows.shape),)
        if getattr(self, "_qproj_key", None) != key:
            weight = torch.cat((params[0], params[2]), 0).contiguous()
            bias = torch.cat((params[1], params[3]), 0).contiguous()
            split = ops.split_weight(weight)
            # the table keeps `pos_rows` referenced so that its memory cannot be handed to other data
            built = (weight, ops.linear_tf32x3(pos_rows, weight, bias, presplit=split), pos_rows, split)
            if _capturing(pos_rows):
                return built[0], built[1], built[3]
            self._qproj, self._qproj_key = built, key
        return self._qproj[0], self._qproj[1], self._qproj[3]

    def forward_shared_pos(self, src, pos, reference_points, input_spatial_shapes, input_level_start_index,
                           value=None, src16=None):
        """`forward(src + pos, reference_points, src, ...)` without forming `src + pos`: the two query
        projections run as ONE GEMM on `src`; the fused kernel reads offsets and logits in place from its
        [N, S, 3*M*L*P] output and adds the cached `pos @ W^T + b` row of the query
        ((src + pos) W^T + b = src W^T + (pos W^T + b)).  `value`: a callable returning the projected value
        [N, S, M, D] (query-range sharding: `src` holds this rank's rows only and the value rows of the other
        ranks are still in flight while the query GEMM runs); default: `project_value(src)`.
        Under a 16-bit autocast (linear="autocast"): the query GEMM and the value projection read `src16`, the 16-bit
        copy of `src` (default: `src` cast), and the 16-bit packed forward adds the same fp32 table."""
        if _resolve(self.linear) == "autocast":
            return self._forward_shared_pos_mixed(src, pos, reference_points, input_spatial_shapes,
                                                  input_level_start_index, value, src16)
        if value is None:
            value = self.project_value(src)
        weight, table, split = self._query_projection(pos[0])
        proj = ops.linear_tf32x3(src, weight, None, presplit=split)
        if callable(value):
            value = value()
        ref = reference_points
        if ref.stride(0) == 0:
            ref = ref[:1]
        out = ops.ms_deform_attn_fused_forward_packed(value, input_spatial_shapes, input_level_start_index,
                                                      ref.contiguous(), proj, self.n_levels, self.n_points,
                                                      query_table=table)
        return _linear(self.output_proj, out, self.linear)

    def _forward_shared_pos_mixed(self, src, pos, reference_points, input_spatial_shapes, input_level_start_index,
                                  value, src16):
        if src16 is None:
            src16 = src.to(_autocast_dtype())
        if value is None:
            value = self.project_value(src16)
        weight, table, _ = self._query_projection(pos[0])
        # the 16-bit query GEMM, cached 16-bit stacked weight; the bias is in the table
        w16 = _weight16_of(weight, self.__dict__, src16.dtype)
        proj = ops.linear_mixed(src16, w16) if ops.linear_mixed_supported(src16, w16) else F.linear(src16, weight)
        if callable(value):
            value = value()
        ref = reference_points
        if ref.stride(0) == 0:
            ref = ref[:1]
        ref = ref.contiguous()
        if ops.ms_deform_attn_fused_mixed_forward_packed_supported(value, ref, proj, self.n_levels, self.n_points,
                                                                   table):
            out = ops.ms_deform_attn_fused_mixed_forward_packed(value, input_spatial_shapes, input_level_start_index,
                                                                ref, proj, self.n_levels, self.n_points,
                                                                query_table=table)
        else:                                              # e.g. a value view the kernel cannot take
            q = src + pos
            return self.forward(q, reference_points, src16, input_spatial_shapes, input_level_start_index)
        return _linear(self.output_proj, out, self.linear)


def _activation(name):
    return {"relu": F.relu, "gelu": F.gelu, "glu": F.glu}[name]


class MSDeformAttnTransformerEncoderLayer(nn.Module):
    """msdeformattn.py:102-142 (post-norm: attention, add & norm, FFN, add & norm)."""

    def __init__(self, d_model=256, d_ffn=1024, dropout=0.1, activation="relu", n_levels=4, n_heads=8,
                 n_points=4, core: Optional[CoreFn] = None, fused: bool = False, linear: str = "torch"):
        super().__init__()
        self.linear = linear
        self.self_attn = MSDeformAttn(d_model, n_levels, n_heads, n_points, core=core, fused=fused, linear=linear)
        self.dropout1 = nn.Dropout(dropout)
        self.norm1 = nn.LayerNorm(d_model)
        self.linear1 = nn.Linear(d_model, d_ffn)
        self.activation = _activation(activation)
        self.dropout2 = nn.Dropout(dropout)
        self.linear2 = nn.Linear(d_ffn, d_model)
        self.dropout3 = nn.Dropout(dropout)
        self.norm2 = nn.LayerNorm(d_model)

    def forward_ffn(self, src):
        p = self.dropout2.p if self.dropout2.training else 0.0
        if (self.activation is F.relu and _resolve(self.linear) == "tf32x3" and torch.is_grad_enabled() and 0.0 < p < 1.0
                and LinearTF32x3Function.supported(src, self.linear1.weight)):
            # training: linear1 + ReLU + dropout2 as one autograd node (one pass over the hidden gradient)
            hidden = LinearTF32x3Function.apply(src, self.linear1.weight, self.linear1.bias, True, p)
        else:
            if self.activation is F.relu:          # ReLU rides in the GEMM epilogue of the tf32x3 kernel
                hidden = _linear(self.linear1, src, self.linear, relu=True)
            else:
                hidden = self.activation(_linear(self.linear1, src, self.linear))
            hidden = self.dropout2(hidden)
        return _add_norm(self.norm2, src, self.dropout3(_linear(self.linear2, hidden, self.linear)), self.linear)

    def forward(self, src, pos, reference_points, spatial_shapes, level_start_index, padding_mask=None):
        return self._forward_pair(src, None, pos, reference_points, spatial_shapes, level_start_index, padding_mask)[0]

    def _forward_pair(self, src, src16, pos, reference_points, spatial_shapes, level_start_index, padding_mask=None):
        """-> (output, its 16-bit copy or None).  `src16`: the 16-bit copy of `src` that the previous layer's mixed
        residual + LayerNorm kernel wrote, or None.  Under a 16-bit autocast with linear="autocast" the two norms go
        through `_add_norm_mixed`, and the GEMMs that read a norm's output (value_proj, linear1, and the next layer's)
        read its copy instead of casting it again; otherwise `forward`'s computation, and no copy."""
        if _resolve(self.linear) != "autocast":
            if self.self_attn.can_fold_pos(src, pos, reference_points, padding_mask):
                attn = self.self_attn.forward_shared_pos(src, pos, reference_points, spatial_shapes, level_start_index)
            else:
                q = src if pos is None else src + pos
                attn = self.self_attn(q, reference_points, src, spatial_shapes, level_start_index, padding_mask)
            return self.forward_ffn(_add_norm(self.norm1, src, self.dropout1(attn), self.linear)), None
        if src16 is None and src.dtype == torch.float32:
            src16 = src.to(_autocast_dtype())              # the first layer's input: a plain cast
        value_in = src16 if src16 is not None else src
        if self.self_attn.can_fold_pos(src, pos, reference_points, padding_mask):
            attn = self.self_attn.forward_shared_pos(src, pos, reference_points, spatial_shapes, level_start_index,
                                                     src16=src16)
        else:
            q = src if pos is None else src + pos
            attn = self.self_attn(q, reference_points, value_in, spatial_shapes, level_start_index, padding_mask)
        y, y16 = _add_norm_mixed(self.norm1, src, self.dropout1(attn))
        return self._forward_ffn_mixed(y, y16)

    def _forward_ffn_mixed(self, src, src16):
        """`forward_ffn` under a 16-bit autocast: linear1 reads `src16` when there is one -> (output, its copy)."""
        x = src16 if src16 is not None else src
        p = self.dropout2.p if self.dropout2.training else 0.0
        hidden = None
        if self.activation is F.relu and torch.is_grad_enabled() and 0.0 < p < 1.0:
            # training: linear1 + ReLU + dropout2 as one autograd node (one pass over the hidden gradient)
            hidden = _linear_mixed(self.linear1, x, relu=True, dropout_p=p)
        if hidden is None:
            if self.activation is F.relu:      # the ReLU rides in the 16-bit GEMM's epilogue
                hidden = _linear(self.linear1, x, self.linear, relu=True)
            else:
                hidden = self.activation(_linear(self.linear1, x, self.linear))
            hidden = self.dropout2(hidden)
        return _add_norm_mixed(self.norm2, src, self.dropout3(_linear(self.linear2, hidden, self.linear)))


_REF_CACHE = ShapeCache()


def reference_points_for(levels: Sequence[Tuple[int, int]], device, dtype=torch.float32):
    """[1, S, L, 2] pixel-centre reference points of every query, replicated over levels, for
    valid_ratios == 1 (msdeformattn.py:152-166 with the all-False masks of :68-69).

    `levels` is a host-side list, so no CUDA tensor is iterated (msdeformattn.py:154 syncs).  The
    points are input-independent: they are computed once per (levels, device, dtype) on the host
    with true IEEE division -- torch's CUDA tensor/scalar division multiplies by a reciprocal and
    lands 1 ulp away from the reference's tensor/tensor division -- and cached on the device."""
    key = (tuple((int(h), int(w)) for h, w in levels), str(device), dtype)
    hit = _REF_CACHE.get(key)
    if hit is None:
        pts = []
        for H, W in key[0]:
            ys = torch.linspace(0.5, H - 0.5, H, dtype=dtype) / torch.tensor(float(H), dtype=dtype)
            xs = torch.linspace(0.5, W - 0.5, W, dtype=dtype) / torch.tensor(float(W), dtype=dtype)
            yy, xx = torch.meshgrid(ys, xs, indexing="ij")
            pts.append(torch.stack((xx.reshape(-1), yy.reshape(-1)), -1))
        ref = torch.cat(pts, 0)
        hit = _REF_CACHE.put(key, ref[None, :, None, :].expand(1, ref.shape[0], len(key[0]), 2).contiguous().to(device))
    return hit


_LEVEL_CACHE = ShapeCache()


def level_tensors_for(levels: Sequence[Tuple[int, int]], device):
    """(spatial_shapes [L, 2], level_start_index [L]) int64 device tensors for a pyramid (msdeformattn.py:82-85),
    built once per (levels, device): they depend only on the shapes, and a host-to-device copy per
    forward would keep the call from being captured in a CUDA graph."""
    key = (tuple((int(h), int(w)) for h, w in levels), str(device))
    hit = _LEVEL_CACHE.get(key)
    if hit is None:
        shapes = torch.tensor(key[0], dtype=torch.long)
        lsi = torch.cat((shapes.new_zeros(1), shapes.prod(1).cumsum(0)[:-1]))
        hit = _LEVEL_CACHE.put(key, (shapes.to(device), lsi.to(device)))
    return hit


class MSDeformAttnTransformerEncoder(nn.Module):
    """msdeformattn.py:145-176."""

    def __init__(self, encoder_layer, num_layers):
        super().__init__()
        self.layers = nn.ModuleList([copy.deepcopy(encoder_layer) for _ in range(num_layers)])
        self.num_layers = num_layers

    @staticmethod
    def get_reference_points(spatial_shapes, valid_ratios, device):
        """Reference signature (msdeformattn.py:152-166); general valid_ratios."""
        levels = [(int(h), int(w)) for h, w in
                  (spatial_shapes.tolist() if torch.is_tensor(spatial_shapes) else spatial_shapes)]
        base = reference_points_for(levels, device)[0, :, 0]            # [S, 2] at ratio 1
        sizes = torch.tensor([h * w for h, w in levels])
        lvl_of = torch.repeat_interleave(torch.arange(len(levels)), sizes).to(device)
        own = valid_ratios[:, lvl_of]                                    # [N, S, 2] ratio of own level
        return (base[None] / own)[:, :, None] * valid_ratios[:, None]    # [N, S, L, 2]

    def forward(self, src, spatial_shapes, level_start_index, valid_ratios, pos=None, padding_mask=None,
                levels: Optional[List[Tuple[int, int]]] = None):
        if levels is not None and valid_ratios is None:
            ref = reference_points_for(levels, src.device).expand(src.shape[0], -1, -1, -1)
        else:
            ref = self.get_reference_points(spatial_shapes, valid_ratios, src.device)
        out, out16 = src, None
        for layer in self.layers:
            if _resolve(layer.linear) == "autocast":
                # under autocast each layer hands the 16-bit copy of its output to the next
                out, out16 = layer._forward_pair(out, out16, pos, ref, spatial_shapes, level_start_index, padding_mask)
            else:
                out = layer(out, pos, ref, spatial_shapes, level_start_index, padding_mask)
        return out


class MSDeformAttnTransformerEncoderOnly(nn.Module):
    """msdeformattn.py:26-99: flattens the per-level maps, adds the level embedding to the position
    embedding and runs the encoder.  Returns (memory, spatial_shapes, level_start_index, valid_ratios)."""

    def __init__(self, d_model=256, nhead=8, num_encoder_layers=6, dim_feedforward=1024, dropout=0.1,
                 activation="relu", num_feature_levels=4, enc_n_points=4, core: Optional[CoreFn] = None,
                 fused: bool = False, linear: str = "torch"):
        super().__init__()
        self.d_model, self.nhead = d_model, nhead
        layer = MSDeformAttnTransformerEncoderLayer(d_model, dim_feedforward, dropout, activation,
                                                    num_feature_levels, nhead, enc_n_points, core=core,
                                                    fused=fused, linear=linear)
        self.encoder = MSDeformAttnTransformerEncoder(layer, num_encoder_layers)
        self.level_embed = nn.Parameter(torch.empty(num_feature_levels, d_model))
        self._reset_parameters()

    def _reset_parameters(self):
        for p in self.parameters():
            if p.dim() > 1:
                nn.init.xavier_uniform_(p)
        for m in self.modules():
            if isinstance(m, MSDeformAttn):
                m._reset_parameters()
        nn.init.normal_(self.level_embed)

    def _level_pos(self, pos_embeds):
        if not torch.is_grad_enabled() and all(p.size(0) == 1 or p.stride(0) == 0 for p in pos_embeds):
            # one embedding for the whole batch (the pixel decoder's mask-free sine embedding): keep ONE copy
            # of the rows and broadcast it, so that callers can tell (batch stride 0)
            n = pos_embeds[0].size(0)
            rows = torch.cat([p[:1].flatten(2).transpose(1, 2) + self.level_embed[i].view(1, 1, -1)
                              for i, p in enumerate(pos_embeds)], 1)
            return rows.expand(n, -1, -1)
        return torch.cat([p.flatten(2).transpose(1, 2) + self.level_embed[i].view(1, 1, -1)
                          for i, p in enumerate(pos_embeds)], 1)

    def flatten_inputs(self, srcs, pos_embeds, src_flat=None, levels=None):
        """`src_flat` / `levels` (not in the reference): the per-level maps already laid out as the concatenated
        [N, S, C] rows (the pixel decoder's fused GroupNorm writes them there), `srcs` is then ignored."""
        if src_flat is None:
            levels = [(int(s.shape[2]), int(s.shape[3])) for s in srcs]
            src = torch.cat([s.flatten(2).transpose(1, 2) for s in srcs], 1)
        else:
            levels = [(int(h), int(w)) for h, w in levels]
            src = src_flat
        if torch.is_grad_enabled():
            pos = self._level_pos(pos_embeds)
        else:
            # inference: position embedding + level embedding depends on the shapes and on one parameter only;
            # built once per (position tensors, level_embed version) instead of on every call (SURVEY 8f.4)
            key = (tuple((p.data_ptr(), _version_of(p), tuple(p.shape), tuple(p.stride())) for p in pos_embeds),
                   self.level_embed.data_ptr(), _version_of(self.level_embed))
            if getattr(self, "_pos_cache_key", None) != key:
                if _capturing(pos_embeds[0]):
                    pos = self._level_pos(pos_embeds)          # not kept: see _capturing
                else:
                    # the position tensors are kept referenced so their memory cannot be handed to other data
                    self._pos_cache_key, self._pos_cache_src = key, list(pos_embeds)
                    self._pos_cache = pos = self._level_pos(pos_embeds)
            else:
                pos = self._pos_cache
        shapes, lsi = level_tensors_for(levels, src.device)
        return src, pos, shapes, lsi, levels

    def forward(self, srcs, pos_embeds, src_flat=None, levels=None):
        src, pos, shapes, lsi, levels = self.flatten_inputs(srcs, pos_embeds, src_flat, levels)
        # masks are all-False in the reference (msdeformattn.py:68-69): valid ratios are exactly 1
        # and the padding mask changes nothing, so neither is materialised
        memory = self.encoder(src, shapes, lsi, None, pos, None, levels=levels)
        valid_ratios = src.new_ones(src.shape[0], len(levels), 2)
        return memory, shapes, lsi, valid_ratios
