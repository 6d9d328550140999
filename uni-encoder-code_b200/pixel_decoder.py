"""Host-side mirror of the reference's ``MSDeformAttnPixelDecoder``
(model/modeling/pixel_decoder/msdeformattn.py:178-386) -- the caller that owns the MSDA hot path:
1x1 input projections + GroupNorm, sine position embedding, the 6-layer deformable encoder, the
per-level split and one FPN level on the stride-4 feature.

Same submodule / parameter names as the reference (``input_proj.{i}.{0,1}``, ``transformer.*``,
``mask_features``, ``adapter_1``, ``layer_1``), so its checkpoints load with ``load_state_dict``.
Constructor arguments are the explicit ones of the reference's ``__init__`` (no detectron2 config
object); ``input_shape`` maps a feature name to ``(channels, stride)``.

Differences, all from SURVEY.md section 8f.4 (input-independent work and host syncs):
* the position embedding of a level depends only on (H, W): computed once per shape / device and
  cached (the reference recomputes it every forward, position_encoding.py:32-55);
* the level split uses the host-side shapes instead of indexing the device-side
  ``level_start_index`` / ``spatial_shapes`` tensors (msdeformattn.py:351-365 -> ``.item()`` syncs).
"""
from __future__ import annotations

import contextlib
import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F
from torch import nn

from . import ops
from .functions import GroupNormFunction, GroupNormRowsFunction
from .modules import CoreFn, MSDeformAttnTransformerEncoderOnly, ShapeCache, _autocast_dtype, _capturing, _resolve


class PositionEmbeddingSine(nn.Module):
    """transformer_decoder/position_encoding.py:15-55 for the mask-free case, cached per shape."""

    def __init__(self, num_pos_feats=64, temperature=10000, normalize=False, scale=None):
        super().__init__()
        if scale is not None and not normalize:
            raise ValueError("normalize should be True if scale is passed")
        self.num_pos_feats, self.temperature, self.normalize = num_pos_feats, temperature, normalize
        self.scale = 2 * math.pi if scale is None else scale
        self._cache = ShapeCache()        # per instance, most recent shapes only

    def _build(self, H, W, device):
        ones = torch.ones((1, H, W), dtype=torch.float32, device=device)
        y_embed, x_embed = ones.cumsum(1), ones.cumsum(2)
        if self.normalize:
            eps = 1e-6
            y_embed = y_embed / (y_embed[:, -1:, :] + eps) * self.scale
            x_embed = x_embed / (x_embed[:, :, -1:] + eps) * self.scale
        dim_t = torch.arange(self.num_pos_feats, dtype=torch.float32, device=device)
        dim_t = self.temperature ** (2 * (dim_t // 2) / self.num_pos_feats)
        px, py = x_embed[:, :, :, None] / dim_t, y_embed[:, :, :, None] / dim_t
        px = torch.stack((px[..., 0::2].sin(), px[..., 1::2].cos()), dim=4).flatten(3)
        py = torch.stack((py[..., 0::2].sin(), py[..., 1::2].cos()), dim=4).flatten(3)
        return torch.cat((py, px), dim=3).permute(0, 3, 1, 2).contiguous()      # [1, 2*npf, H, W]

    def forward(self, x, mask=None):
        if mask is not None:
            raise NotImplementedError("the pixel decoder never passes a mask (msdeformattn.py:345)")
        key = (x.shape[2], x.shape[3], str(x.device))
        pos = self._cache.get(key)
        if pos is None:
            pos = self._build(x.shape[2], x.shape[3], x.device)
            if not _capturing(x):                      # built during a graph capture: not materialised yet, not kept
                self._cache.put(key, pos)
        return pos.expand(x.shape[0], -1, -1, -1)


class _ConvNormAct(nn.Conv2d):
    """Conv2d followed by an optional norm and activation (what detectron2.layers.Conv2d does for
    the reference's lateral / output convolutions, msdeformattn.py:286-300)."""

    def __init__(self, *args, norm=None, activation=None, **kwargs):
        super().__init__(*args, **kwargs)
        self.norm, self.activation = norm, activation

    def forward(self, x, up=None, fused_norm=False, out_dtype=None):
        """conv -> norm -> activation (-> + bilinear up-sampling of `up`, the FPN top-down add of
        msdeformattn.py:372-376).  `fused_norm` (GroupNorm): the norm, the ReLU and the up-sampled add through
        `_group_norm`; `out_dtype` (under torch.autocast, the convolution's 16-bit type): the result rounded to it, the
        copy the next convolution reads."""
        x = super().forward(x)
        if fused_norm and isinstance(self.norm, nn.GroupNorm) and self.activation in (None, F.relu):
            return _group_norm(self.norm, x, relu=self.activation is F.relu, up=up,
                               out_dtype=out_dtype if x.dtype == out_dtype else None)
        if self.norm is not None:
            x = self.norm(x)
        x = x if self.activation is None else self.activation(x)
        if up is not None:
            x = x + F.interpolate(up, size=x.shape[-2:], mode="bilinear", align_corners=False)
        return x


def _group_norm(norm: nn.GroupNorm, x, relu=False, up=None, channel_bias=None, out_dtype=None):
    """``norm(x + channel_bias[None, :, None, None])`` [-> ReLU] [+ bilinear up-sampling of `up`] (`channel_bias`: the
    bias of the convolution that produced x and ran without it).  Where ops.group_norm_supported holds, one statistics
    + one apply kernel (SURVEY 8f.4): ops.group_norm with autograd off, GroupNormFunction, whose backward also runs on
    the library's kernels, with it on; torch otherwise.  A 16-bit x (torch.autocast) gives an fp32 result, or with
    `out_dtype=x.dtype` and the kernels its 16-bit copy."""
    if ops.group_norm_supported(x, norm, up):
        if not torch.is_grad_enabled():
            return ops.group_norm(x, norm, relu=relu, up=up, channel_bias=channel_bias, out_dtype=out_dtype)
        return GroupNormFunction.apply(x, norm.weight, norm.bias, channel_bias, up, norm.num_groups, norm.eps, relu,
                                       out_dtype)
    x = norm(x if channel_bias is None else x + channel_bias.view(1, -1, 1, 1))
    x = F.relu(x) if relu else x
    if up is not None:
        x = x + F.interpolate(up, size=x.shape[-2:], mode="bilinear", align_corners=False)
    return x


def _norm(kind, channels):
    if kind in (None, ""):
        return None
    if kind == "GN":
        return nn.GroupNorm(32, channels)
    raise NotImplementedError(f"norm {kind!r}")


def _c2_xavier_fill(m):
    nn.init.kaiming_uniform_(m.weight, a=1)
    if m.bias is not None:
        nn.init.constant_(m.bias, 0)


class MSDeformAttnPixelDecoder(nn.Module):
    def __init__(self, input_shape: Dict[str, Tuple[int, int]], *, transformer_dropout: float,
                 transformer_nheads: int, transformer_dim_feedforward: int, transformer_enc_layers: int,
                 conv_dim: int, mask_dim: int, norm: Optional[str] = None,
                 transformer_in_features: Sequence[str], common_stride: int,
                 core: Optional[CoreFn] = None, fused: bool = False, linear: str = "torch", amp: bool = False):
        """`amp=True` (not in the reference): `forward_features` runs inside the caller's torch.autocast context
        instead of disabling it -- torch's 16-bit GEMMs and convolutions, and the mixed-precision MSDA op
        (functions.MSDeformAttnMixedFunction; with `fused=True` the 16-bit fused-producer kernels,
        functions.MSDeformAttnFusedFunction, which take the softmax and the location arithmetic off torch).
        `amp=False` is the reference's behaviour: autocast off, fp32.
        `linear="autocast"` (not in the reference): `linear="tf32x3"` where no bf16 / fp16 autocast is active (with
        `amp=False` always); under one, torch's autocast GEMMs and convolutions as with `linear="torch"`, with the
        encoder's residual + LayerNorm steps and the batch-shared position embedding's query projection on the
        mixed-precision kernels (modules._add_norm_mixed, MSDeformAttn.forward_shared_pos), and the five GroupNorms
        on the 16-bit GroupNorm kernels, as `linear="tf32x3"` routes them: the input projections' convolutions run
        without their bias and the rows kernels write the fp32 encoder input, adding it in fp32; the FPN lateral and
        output GroupNorms (with the up-sampled fp32 encoder level, the ReLU) return the 16-bit copy the next
        convolution reads; in inference `mask_features` adds its bias to its 16-bit output in one pass."""
        if amp and linear == "tf32x3":
            raise ValueError('amp=True cannot be combined with linear="tf32x3": the 3xTF32 GEMMs and the fp32 '
                             'GroupNorm / LayerNorm kernels are fp32 paths that autocast would bypass')
        super().__init__()
        self.amp = amp
        by_stride = sorted(input_shape.items(), key=lambda kv: kv[1][1])
        self.in_features = [k for k, _ in by_stride]
        self.feature_channels = [v[0] for _, v in by_stride]
        tr = [(k, v) for k, v in by_stride if k in transformer_in_features]
        self.transformer_in_features = [k for k, _ in tr]
        self.transformer_feature_strides = [v[1] for _, v in tr]
        self.transformer_num_feature_levels = len(tr)
        chans = [v[0] for _, v in tr]
        chans = chans[::-1] if len(tr) > 1 else chans[-1:]          # low -> high resolution
        self.input_proj = nn.ModuleList(
            nn.Sequential(nn.Conv2d(c, conv_dim, kernel_size=1), nn.GroupNorm(32, conv_dim)) for c in chans)
        for proj in self.input_proj:
            nn.init.xavier_uniform_(proj[0].weight, gain=1)
            nn.init.constant_(proj[0].bias, 0)
        self.transformer = MSDeformAttnTransformerEncoderOnly(
            d_model=conv_dim, dropout=transformer_dropout, nhead=transformer_nheads,
            dim_feedforward=transformer_dim_feedforward, num_encoder_layers=transformer_enc_layers,
            num_feature_levels=self.transformer_num_feature_levels, core=core, fused=fused, linear=linear)
        self.pe_layer = PositionEmbeddingSine(conv_dim // 2, normalize=True)
        self.linear = linear
        self.mask_dim = mask_dim
        self.mask_features = nn.Conv2d(conv_dim, mask_dim, kernel_size=1, stride=1, padding=0)
        _c2_xavier_fill(self.mask_features)
        self.oneformer_num_feature_levels = 3
        self.common_stride = common_stride
        self.num_fpn_levels = int(math.log2(min(self.transformer_feature_strides)) - math.log2(common_stride))
        lateral, output = [], []
        use_bias = norm == ""
        for idx, c in enumerate(self.feature_channels[:self.num_fpn_levels]):
            lat = _ConvNormAct(c, conv_dim, kernel_size=1, bias=use_bias, norm=_norm(norm, conv_dim))
            out = _ConvNormAct(conv_dim, conv_dim, kernel_size=3, stride=1, padding=1, bias=use_bias,
                               norm=_norm(norm, conv_dim), activation=F.relu)
            _c2_xavier_fill(lat)
            _c2_xavier_fill(out)
            self.add_module(f"adapter_{idx + 1}", lat)
            self.add_module(f"layer_{idx + 1}", out)
            lateral.append(lat)
            output.append(out)
        self.lateral_convs, self.output_convs = lateral[::-1], output[::-1]

    def forward_features(self, features: Dict[str, torch.Tensor]):
        """-> (mask_features [N, mask_dim, H/4, W/4], lowest-resolution map, 3 multi-scale maps),
        as msdeformattn.py:336-386 (autocast disabled, inputs promoted to fp32; with `amp`, under the caller's
        autocast, if any)."""
        device_type = next(iter(features.values())).device.type
        with contextlib.nullcontext() if self.amp else torch.autocast(device_type=device_type, enabled=False):
            # the inference kernels of SURVEY 8f.3 / 8f.4 (linear="autocast": when no 16-bit autocast is active), and
            # the GroupNorm kernels on the 16-bit maps of the convolutions under one (DESIGN.md 11.3)
            fused_norm = _resolve(self.linear) in ("tf32x3", "autocast")
            out16 = _autocast_dtype() if _resolve(self.linear) == "autocast" else None
            names = self.transformer_in_features[::-1]
            levels = [(int(features[k].shape[2]), int(features[k].shape[3])) for k in names]
            srcs, src_flat = self._input_proj([features[k].float() for k in names], levels, fused_norm)
            pos = [self.pe_layer(features[k]) for k in names]
            memory, _, _, _ = self.transformer(srcs, pos, src_flat=src_flat, levels=levels)
            n = memory.shape[0]
            out: List[torch.Tensor] = [z.transpose(1, 2).reshape(n, -1, h, w) for z, (h, w) in
                                       zip(memory.split([h * w for h, w in levels], dim=1), levels)]
            for idx, name in enumerate(self.in_features[:self.num_fpn_levels][::-1]):
                y = self.lateral_convs[idx](features[name].float(), up=self._nchw(out[-1], memory, fused_norm),
                                            fused_norm=fused_norm, out_dtype=out16)
                out.append(self.output_convs[idx](y, fused_norm=fused_norm, out_dtype=out16))
            return self._mask_features(out[-1], fused_norm), out[0], out[:self.oneformer_num_feature_levels]

    def _input_proj(self, xs, levels, fused_norm):
        """The input projections of the encoder's levels -> (srcs, None): the per-level NCHW maps, which the encoder
        concatenates; or (None, src_flat): that concatenated [N, S, C] tensor, written directly.  With `fused_norm` the
        convolutions run without their bias (torch adds it in a separate pass over the map) and the GroupNorms add it
        on the fly.  When ops.group_norm_rows_supported holds for every level, each level's GroupNorm writes its rows
        of src_flat (no transposing `cat`): ops.group_norm_rows with autograd off, ONE GroupNormRowsFunction node for
        all levels with it on.  Otherwise every level goes through `_group_norm`.  Under torch.autocast the
        convolutions write 16-bit maps and src_flat stays fp32."""
        if not fused_norm:
            return [proj[1](proj[0](x)) for proj, x in zip(self.input_proj, xs)], None
        convs, norms = [proj[0] for proj in self.input_proj], [proj[1] for proj in self.input_proj]
        ys = [F.conv2d(x, c.weight, None, c.stride, c.padding, c.dilation, c.groups) for c, x in zip(convs, xs)]
        starts = [0]
        for h, w in levels:
            starts.append(starts[-1] + h * w)
        src_flat = ys[0].new_empty((ys[0].shape[0], starts[-1], ys[0].shape[1]), dtype=torch.float32)
        rows = [src_flat[:, a:b] for a, b in zip(starts, starts[1:])]
        if not (all(ops.group_norm_rows_supported(y, n, r) for y, n, r in zip(ys, norms, rows))
                and len({(n.num_groups, n.eps) for n in norms}) == 1):
            return [_group_norm(n, y, channel_bias=c.bias) for n, y, c in zip(norms, ys, convs)], None
        if not torch.is_grad_enabled():
            for y, n, c, r in zip(ys, norms, convs, rows):
                ops.group_norm_rows(y, n, r, channel_bias=c.bias)
            return None, src_flat
        del src_flat, rows                             # GroupNormRowsFunction allocates its own output
        return None, GroupNormRowsFunction.apply(norms[0].num_groups, norms[0].eps,
                                                 *[t for y, n, c in zip(ys, norms, convs)
                                                   for t in (y, n.weight, n.bias, c.bias)])

    @staticmethod
    def _nchw(view, memory, fused_norm):
        """Contiguous NCHW copy of a level of the encoder memory (`view` = [N, C, H, W] strided over the
        [N, S, C] memory): one [pixels, C] -> [C, pixels] transpose kernel per image in inference."""
        if view.is_contiguous():
            return view
        n, c, h, w = view.shape
        if not (fused_norm and not torch.is_grad_enabled() and view.is_cuda and view.dtype == torch.float32
                and view.stride(1) == 1 and view.stride(3) == c and view.stride(2) == w * c):
            return view.contiguous()
        dst = torch.empty((n, c, h, w), dtype=view.dtype, device=view.device)
        for i in range(n):
            # view[i] is the transpose of the contiguous [h*w, c] block of rows of image i
            rows = torch.as_strided(view, (h * w, c), (c, 1), view[i].storage_offset())
            ops.transpose2d(rows, out=dst[i])
        return dst

    def _mask_features(self, x, fused_norm):
        conv = self.mask_features
        if fused_norm and not torch.is_grad_enabled() and conv.bias is not None:
            y = F.conv2d(x, conv.weight, None, conv.stride, conv.padding, conv.dilation, conv.groups)
            if ops.channel_bias_supported(y, conv.bias):
                return ops.add_channel_bias_(y, conv.bias)
            return (y + conv.bias.view(1, -1, 1, 1)).to(y.dtype)
        return conv(x)
