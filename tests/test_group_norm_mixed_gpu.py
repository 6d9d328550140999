"""The 16-bit GroupNorm kernels (torch.autocast: the decoder's convolutions write bf16 / fp16 maps).

Kernel contracts, bit for bit, against the fp32 kernels fed the widened map:
* forward: y and mean_rstd == the fp32 train kernel's on x.float(); y16 == y.to(dtype); the rows forward's fp32 rows
  == the fp32 rows kernel's;
* backward: grad_x == the fp32 backward's grad_x (on the widened gradient and x.float()) rounded once; the weight,
  bias, channel-bias and up-sampled-map gradients (fp32) == the fp32 backward's;
* channel bias in place: (x.float() + bias).to(dtype).
Functions are held to torch's autocast composition (widen -> F.group_norm -> [relu] -> [+ interpolate] -> [cast]) under
autograd; the pixel decoder under autocast with the kernels on against the same module with the predicates refusing
16-bit maps.
"""
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from test_autocast_encoder_gpu import ERR_NULL, ERR_UNSUPPORTED, _perturbed, same16
from test_group_norm_train_gpu import CASES, EPS, LEVELS, _full_width_decoder, _inputs
from test_mixed_precision_gpu import deterministic_mode
from test_pixel_decoder import PD_KW, PD_SHAPES, build

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DTYPES = [torch.bfloat16, torch.float16]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _case(shape, groups, up, with_cb, dtype, seed):
    x, w, b, cb, u, cot = _inputs(shape, groups, up, with_cb, seed)
    return x.to(dtype), w, b, cb, u, cot


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _equal_bits(a, b):
    """Equal element for element, NaN where the other is NaN."""
    assert a.dtype == b.dtype
    if a.dtype in DTYPES:
        same16(a, b)
    else:
        assert torch.equal(a.isnan(), b.isnan())
        assert torch.equal(torch.nan_to_num(a, nan=0.0), torch.nan_to_num(b, nan=0.0))


# ---------------------------------------------------------------- forward
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape,groups,relu,up", CASES)
@pytest.mark.parametrize("with_cb", [False, True])
def test_forward_bit_identical_to_fp32_on_the_widened_map(pkg, dtype, shape, groups, relu, up, with_cb):
    x, w, b, cb, u, _ = _case(shape, groups, up, with_cb, dtype, seed=sum(shape) + groups)
    ref, ref_stats = pkg.ops.group_norm_train(x.float(), w, b, groups, EPS, relu=relu, up=u, channel_bias=cb)
    n0 = pkg.launch_count()
    y, stats = pkg.ops.group_norm_train(x, w, b, groups, EPS, relu=relu, up=u, channel_bias=cb)
    y16, stats16 = pkg.ops.group_norm_train(x, w, b, groups, EPS, relu=relu, up=u, channel_bias=cb, out_dtype=dtype)
    assert pkg.launch_count() - n0 == 4
    assert y.dtype == torch.float32 and y16.dtype == dtype
    assert torch.equal(y, ref) and torch.equal(stats, ref_stats) and torch.equal(stats16, ref_stats)
    same16(y16, ref.to(dtype))
    norm = torch.nn.GroupNorm(groups, shape[1], eps=EPS).to(DEV)
    with torch.no_grad():
        norm.weight.copy_(w)
        norm.bias.copy_(b)
    assert pkg.ops.group_norm_supported(x, norm, u)
    assert torch.equal(pkg.ops.group_norm(x, norm, relu=relu, up=u, channel_bias=cb), ref)
    same16(pkg.ops.group_norm(x, norm, relu=relu, up=u, channel_bias=cb, out_dtype=dtype), y16)
    # both outputs in one call of the C entry
    N, C, H, W = shape
    both, both16 = torch.empty_like(ref), torch.empty_like(x)
    ws = torch.empty(int(pkg._lib.lib.msda_b200_group_norm_workspace_bytes(N, groups)), dtype=torch.uint8, device=DEV)
    rc = pkg.ops._GN_MIXED[dtype]["group_norm_nchw_mixed"](
        x.data_ptr(), pkg.ops._ptr(cb), w.data_ptr(), b.data_ptr(), both.data_ptr(), both16.data_ptr(), N, C, H, W,
        groups, EPS, int(relu), pkg.ops._ptr(u), u.size(2) if u is not None else 0, u.size(3) if u is not None else 0,
        ws.data_ptr(), _stream())
    assert rc == 0
    assert torch.equal(both, ref)
    same16(both16, y16)


@pytest.mark.parametrize("dtype", DTYPES)
def test_rows_forward_bit_identical_into_a_slice(pkg, dtype):
    groups = 32
    N, C = LEVELS[0][0][:2]
    sizes = [s[2] * s[3] for s, _ in LEVELS]
    wide = torch.full((N, sum(sizes) + 9, C), -7.0, device=DEV)
    ref = torch.full_like(wide, -7.0)
    start = 4
    for i, (shape, with_cb) in enumerate(LEVELS):
        x, w, b, cb, _, _ = _case(shape, groups, None, with_cb, dtype, seed=i + 11)
        hw = shape[2] * shape[3]
        n0 = pkg.launch_count()
        stats = pkg.ops.group_norm_rows_train(x, w, b, groups, EPS, wide[:, start:start + hw], channel_bias=cb)
        assert pkg.launch_count() - n0 == 2
        want = pkg.ops.group_norm_rows_train(x.float(), w, b, groups, EPS, ref[:, start:start + hw], channel_bias=cb)
        assert torch.equal(stats, want)
        start += hw
    assert torch.equal(wide, ref)                  # the rows and, untouched, everything around them


# ---------------------------------------------------------------- backward
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape,groups,relu,up", CASES)
@pytest.mark.parametrize("with_cb", [False, True])
@pytest.mark.parametrize("grad16", [False, True])
def test_backward_bit_identical_to_fp32_on_the_widened_inputs(pkg, dtype, shape, groups, relu, up, with_cb, grad16):
    x, w, b, cb, u, cot = _case(shape, groups, up, with_cb, dtype, seed=sum(shape) + 7)
    _, stats = pkg.ops.group_norm_train(x, w, b, groups, EPS, relu=relu, up=u, channel_bias=cb)
    g = cot.to(dtype) if grad16 else cot
    kw = dict(relu=relu, channel_bias=cb, up_shape=tuple(u.shape[-2:]) if u is not None else None,
              with_channel_bias=with_cb)
    ref = pkg.ops.group_norm_backward(g.float(), x.float(), w, b, stats, groups, **kw)
    n0 = pkg.launch_count()
    got = pkg.ops.group_norm_backward(g, x, w, b, stats, groups, **kw)
    assert pkg.launch_count() - n0 == 3 + (u is not None)
    again = pkg.ops.group_norm_backward(g, x, w, b, stats, groups, **kw)
    assert got[0].dtype == dtype
    same16(got[0], ref[0].to(dtype))
    for name, a, r, a2 in zip(("weight", "bias", "channel_bias", "up"), got[1:], ref[1:], again[1:]):
        if r is None:
            assert a is None, name
            continue
        assert a.dtype == torch.float32 and torch.equal(a, r) and torch.equal(a, a2), name
    same16(got[0], again[0])


@pytest.mark.parametrize("dtype", DTYPES)
def test_rows_backward_bit_identical(pkg, dtype):
    groups = 32
    for i, (shape, with_cb) in enumerate(LEVELS):
        x, w, b, cb, _, cot = _case(shape, groups, None, with_cb, dtype, seed=i + 21)
        N, C, H, W = shape
        rows = torch.empty(N, H * W, C, device=DEV)
        stats = pkg.ops.group_norm_rows_train(x, w, b, groups, EPS, rows, channel_bias=cb)
        wide = torch.randn(N, H * W + 6, C, device=DEV)
        grad_rows = wide[:, 3:3 + H * W]                               # a slice of a wider gradient
        ref = pkg.ops.group_norm_rows_backward(grad_rows, x.float(), w, b, stats, groups, channel_bias=cb,
                                               with_channel_bias=with_cb)
        n0 = pkg.launch_count()
        got = pkg.ops.group_norm_rows_backward(grad_rows, x, w, b, stats, groups, channel_bias=cb,
                                               with_channel_bias=with_cb)
        assert pkg.launch_count() - n0 == 3
        same16(got[0], ref[0].to(dtype))
        for a, r in zip(got[1:], ref[1:]):
            assert (a is None and r is None) or torch.equal(a, r)


# ---------------------------------------------------------------- functions against torch's autocast composition
def _composition_grads(x16, w, b, cb, u, groups, relu, out_dtype, cot):
    leaves = [t.detach().clone().requires_grad_(True) if t is not None else None for t in (x16, w, b, cb, u)]
    x, ww, bb, c, uu = leaves
    z = x.float() if c is None else x.float() + c.view(1, -1, 1, 1)
    y = F.group_norm(z, groups, ww, bb, EPS)
    y = torch.relu(y) if relu else y
    if uu is not None:
        y = y + F.interpolate(uu, size=x.shape[-2:], mode="bilinear", align_corners=False)
    y = y.to(out_dtype) if out_dtype is not None else y
    (y.float() * cot).sum().backward()
    return y.detach(), [t.grad if t is not None else None for t in leaves]


def _within_one_rounding(a, r, dtype):
    """|a - r| <= one 16-bit unit in the last place at max |r| (plus that of each element)."""
    unit = 2.0 ** -8 if dtype == torch.bfloat16 else 2.0 ** -11
    bound = unit * (r.float().abs() + r.float().abs().max())
    assert bool(((a.float() - r.float()).abs() <= bound).all()), (a.float() - r.float()).abs().max().item()


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape,groups,relu,up", [CASES[1], CASES[2], CASES[7]])
@pytest.mark.parametrize("out16", [False, True])
def test_group_norm_function_matches_the_autocast_composition(pkg, dtype, shape, groups, relu, up, out16):
    x, w, b, cb, u, cot = _case(shape, groups, up, True, dtype, seed=3)
    out_dtype = dtype if out16 else None
    leaves = [t.clone().requires_grad_(True) for t in (x, w, b, cb)] + [u.clone().requires_grad_(True) if u is not None
                                                                       else None]
    y = pkg.GroupNormFunction.apply(*leaves, groups, EPS, relu, out_dtype)
    assert y.dtype == (dtype if out16 else torch.float32)
    (y.float() * cot).sum().backward()
    ref_y, ref_g = _composition_grads(x, w, b, cb, u, groups, relu, out_dtype, cot)
    _within_one_rounding(y.detach(), ref_y, dtype)
    assert leaves[0].grad.dtype == dtype
    _within_one_rounding(leaves[0].grad, ref_g[0], dtype)
    for t, r in zip(leaves[1:], ref_g[1:]):
        if r is not None:
            assert t.grad.dtype == torch.float32
            assert (t.grad - r).abs().max().item() <= 1e-4 * r.abs().max().item() + 1e-6


@pytest.mark.parametrize("dtype", DTYPES)
def test_group_norm_function_honours_needs_input_grad(pkg, dtype):
    x, w, b, cb, u, cot = _case((2, 64, 8, 12), 32, (4, 6), True, dtype, seed=4)
    xs = x.clone().requires_grad_(True)
    y = pkg.GroupNormFunction.apply(xs, w, b, cb, u, 32, EPS, True, dtype)
    (y.float() * cot).sum().backward()
    assert xs.grad is not None and xs.grad.dtype == dtype
    ws = w.clone().requires_grad_(True)
    us = u.clone().requires_grad_(True)
    n0 = pkg.launch_count()
    y = pkg.GroupNormFunction.apply(x, ws, b, cb, us, 32, EPS, False)
    (y * cot).sum().backward()
    assert pkg.launch_count() - n0 == 2 + 4
    assert ws.grad is not None and us.grad is not None and us.grad.dtype == torch.float32


@pytest.mark.parametrize("dtype", DTYPES)
def test_group_norm_rows_function_matches_the_autocast_composition(pkg, dtype):
    groups = 32
    per_level = [_case(shape, groups, None, cb, dtype, seed=i + 31) for i, (shape, cb) in enumerate(LEVELS)]
    N, C = LEVELS[0][0][:2]
    S = sum(s[2] * s[3] for s, _ in LEVELS)
    cot = torch.randn(N, S, C, device=DEV)
    leaves = [[t.clone().requires_grad_(True) if t is not None else None for t in p[:4]] for p in per_level]
    out = pkg.GroupNormRowsFunction.apply(groups, EPS, *[t for lv in leaves for t in lv])
    assert out.dtype == torch.float32
    (out * cot).sum().backward()
    ref_leaves = [[t.clone().requires_grad_(True) if t is not None else None for t in p[:4]] for p in per_level]
    ref = torch.cat([F.group_norm(x.float() + (cb.view(1, -1, 1, 1) if cb is not None else 0), groups, w, b, EPS)
                     .flatten(2).transpose(1, 2) for x, w, b, cb in ref_leaves], 1)
    (ref * cot).sum().backward()
    _within_one_rounding(out.detach(), ref.detach(), dtype)
    for lv, rv in zip(leaves, ref_leaves):
        assert lv[0].grad.dtype == dtype
        _within_one_rounding(lv[0].grad, rv[0].grad, dtype)
        for t, r in zip(lv[1:], rv[1:]):
            if r is not None:
                assert (t.grad - r.grad).abs().max().item() <= 1e-4 * r.grad.abs().max().item() + 1e-6
    mixed = [leaves[0][0].detach().float()] + leaves[0][1:] + [t.detach() for t in leaves[1]]
    with pytest.raises(RuntimeError, match="one dtype"):
        pkg.GroupNormRowsFunction.apply(groups, EPS, *mixed)


# ---------------------------------------------------------------- edge cases
def test_fp16_overflow_gives_inf(pkg):
    x, w, b, cb, u, cot = _case((1, 64, 8, 8), 32, None, False, torch.float16, seed=6)
    big = b + 1e5                                                      # every output beyond the fp16 range
    y16, stats = pkg.ops.group_norm_train(x, w, big, 32, EPS, out_dtype=torch.float16)
    ref, _ = pkg.ops.group_norm_train(x.float(), w, big, 32, EPS)
    assert bool(torch.isinf(y16).any())
    same16(y16, ref.to(torch.float16))
    g = cot * 1e6                                                      # grad_x beyond the fp16 range
    got = pkg.ops.group_norm_backward(g, x, w * 100, b, stats, 32)
    want = pkg.ops.group_norm_backward(g, x.float(), w * 100, b, stats, 32)
    assert bool(torch.isinf(got[0]).any())
    same16(got[0], want[0].to(torch.float16))


@pytest.mark.parametrize("dtype", DTYPES)
def test_non_finite_inputs(pkg, dtype):
    x, w, b, cb, u, cot = _case((2, 64, 8, 8), 32, (4, 4), True, dtype, seed=8)
    x[0, 0, 1, 1] = float("nan")
    x[1, 5, 2, 3] = float("inf")
    y, stats = pkg.ops.group_norm_train(x, w, b, 32, EPS, up=u, channel_bias=cb)
    ref, ref_stats = pkg.ops.group_norm_train(x.float(), w, b, 32, EPS, up=u, channel_bias=cb)
    _equal_bits(y, ref)
    _equal_bits(stats, ref_stats)
    got = pkg.ops.group_norm_backward(cot, x, w, b, stats, 32, channel_bias=cb, up_shape=(4, 4))
    want = pkg.ops.group_norm_backward(cot, x.float(), w, b, stats, 32, channel_bias=cb, up_shape=(4, 4))
    _equal_bits(got[0], want[0].to(dtype))
    for a, r in zip(got[1:], want[1:]):
        if r is not None:
            _equal_bits(a, r)


@pytest.mark.parametrize("dtype", DTYPES)
def test_misaligned_view_and_output_pointer_rules(pkg, dtype):
    N, C, H, W, groups = 1, 64, 6, 8, 32
    x, w, b, _, _, cot = _case((N, C, H, W), groups, None, False, dtype, seed=9)
    flat = torch.empty(x.numel() + 1, dtype=dtype, device=DEV)
    view = flat[1:].view(x.shape)                                      # a 2-byte offset
    view.copy_(x)
    norm = torch.nn.GroupNorm(groups, C, eps=EPS).to(DEV)
    assert not pkg.ops.group_norm_supported(view, norm)
    assert not pkg.ops.group_norm_rows_supported(view, norm, torch.empty(N, H * W, C, device=DEV))
    assert not pkg.ops.channel_bias_supported(view, w)
    entries = pkg.ops._GN_MIXED[dtype]
    ws = torch.empty(int(pkg._lib.lib.msda_b200_group_norm_backward_workspace_bytes(N, C)), dtype=torch.uint8,
                     device=DEV)
    y = torch.empty(x.shape, device=DEV)
    y16 = torch.empty_like(x)
    tail = (N, C, H, W, groups, EPS, 0, None, 0, 0, ws.data_ptr(), _stream())
    assert entries["group_norm_nchw_mixed"](view.data_ptr(), None, w.data_ptr(), b.data_ptr(), y.data_ptr(), None,
                                            *tail) == ERR_UNSUPPORTED
    assert entries["group_norm_nchw_mixed"](x.data_ptr(), None, w.data_ptr(), b.data_ptr(), None, None,
                                            *tail) == ERR_NULL
    stats = torch.empty(N, groups, 2, device=DEV)
    assert entries["group_norm_nchw_mixed_train"](x.data_ptr(), None, w.data_ptr(), b.data_ptr(), None,
                                                  y16.data_ptr(), None, *tail) == ERR_NULL
    assert entries["group_norm_nchw_mixed_train"](x.data_ptr(), None, w.data_ptr(), b.data_ptr(), None,
                                                  y16.data_ptr(), stats.data_ptr(), *tail) == 0
    assert entries["group_norm_nchw_to_rows_mixed"](view.data_ptr(), None, w.data_ptr(), b.data_ptr(), y.data_ptr(),
                                                    C, H * W * C, N, C, H * W, groups, EPS, 0, ws.data_ptr(),
                                                    _stream()) == ERR_UNSUPPORTED
    g16 = cot.to(dtype)
    gx = torch.empty_like(x)
    gw, gb = torch.empty_like(w), torch.empty_like(b)
    bwd = entries["group_norm_backward_nchw_mixed"]
    rest = (None, w.data_ptr(), b.data_ptr(), stats.data_ptr(), gx.data_ptr(), gw.data_ptr(), gb.data_ptr(), None,
            None, N, C, H, W, groups, 0, 0, 0, ws.data_ptr(), _stream())
    assert bwd(cot.data_ptr(), g16.data_ptr(), x.data_ptr(), *rest) == ERR_UNSUPPORTED          # both gradients
    assert bwd(None, None, x.data_ptr(), *rest) == ERR_NULL                                     # neither
    assert bwd(None, g16.data_ptr(), view.data_ptr(), *rest) == ERR_UNSUPPORTED                 # x at 2 bytes
    assert bwd(None, g16.data_ptr(), x.data_ptr(), *rest) == 0
    assert entries["group_norm_rows_backward_mixed"](
        torch.randn(N, H * W, C, device=DEV).data_ptr(), C, H * W * C, view.data_ptr(), None, w.data_ptr(),
        b.data_ptr(), stats.data_ptr(), gx.data_ptr(), gw.data_ptr(), gb.data_ptr(), None, N, C, H * W, groups, 0,
        ws.data_ptr(), _stream()) == ERR_UNSUPPORTED
    assert entries["add_channel_bias_nchw"](view.data_ptr(), w.data_ptr(), N, C, H * W, _stream()) == ERR_UNSUPPORTED
    assert entries["add_channel_bias_nchw"](None, w.data_ptr(), N, C, H * W, _stream()) == ERR_NULL
    with pytest.raises(RuntimeError, match="out_dtype"):
        pkg.ops.group_norm_train(x, w, b, groups, EPS, out_dtype=torch.float16 if dtype == torch.bfloat16
                                 else torch.bfloat16)


@pytest.mark.parametrize("dtype", DTYPES)
def test_channel_bias_in_place(pkg, dtype):
    gen = torch.Generator().manual_seed(12)
    x = (torch.randn(3, 40, 6, 12, generator=gen) * 4).to(dtype).to(DEV)
    bias = (torch.randn(40, generator=gen) * 3).to(DEV)
    want = (x.float() + bias.view(1, -1, 1, 1)).to(dtype)
    n0 = pkg.launch_count()
    got = pkg.ops.add_channel_bias_(x, bias)
    assert pkg.launch_count() - n0 == 1 and got.data_ptr() == x.data_ptr()
    same16(got, want)


# ---------------------------------------------------------------- the pixel decoder under autocast
def _refuse16(mp, pkg):
    """Patch the predicates to refuse 16-bit maps: the decoder's autocast path then takes torch's GroupNorms."""
    for name in ("group_norm_supported", "group_norm_rows_supported", "channel_bias_supported"):
        real = getattr(pkg.ops, name)
        mp.setattr(pkg.ops, name, lambda x, *a, _real=real, **k: x.dtype == torch.float32 and _real(x, *a, **k))


def _step(pkg, m, feats, cots, dtype):
    leaves = {k: v.clone().requires_grad_(True) for k, v in feats.items()}
    m.zero_grad(set_to_none=True)
    n0 = pkg.launch_count()
    with torch.autocast("cuda", dtype=dtype):
        mask, low, multi = m.forward_features(leaves)
    fwd = pkg.launch_count() - n0
    loss = sum((o.float() * c).sum() for o, c in zip([mask, low, *multi], cots))
    n0 = pkg.launch_count()
    loss.backward()
    bwd = pkg.launch_count() - n0
    grads = {n: p.grad.float().clone() for n, p in m.named_parameters() if p.grad is not None}
    grads.update({"feat::" + k: v.grad.float().clone() for k, v in leaves.items()})
    return [o.detach().float() for o in (mask, low, *multi)], grads, fwd, bwd


FULL_SHAPES = {"res2": (96, 4), "res3": (192, 8), "res4": (384, 16), "res5": (768, 32)}     # _full_width_decoder's
FULL_KW = dict(transformer_dropout=0.0, transformer_nheads=8, transformer_dim_feedforward=1024, transformer_enc_layers=2,
               conv_dim=256, mask_dim=256, norm="GN", transformer_in_features=["res3", "res4", "res5"], common_stride=4)


def _autocast_twin(pkg, m, shapes, kw):
    """`m` rebuilt with amp=True, linear="autocast" and the same parameters."""
    twin = pkg.pixel_decoder.MSDeformAttnPixelDecoder(shapes, fused=True, linear="autocast", amp=True, **kw)
    twin.load_state_dict(m.state_dict())
    return twin.to(DEV)


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def _on_and_off(pkg, m, feats, dtype, monkeypatch):
    """Inference forward and a training step with the 16-bit kernels on and off, and the off step on features moved
    by one 16-bit unit (the spread to expect), each held to that spread -> (the GroupNorm ops the inference forward
    called, sorted; training launches on - off: forward, backward)."""
    flags = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.deterministic)
    torch.backends.cudnn.deterministic = True
    try:
        calls = []
        with monkeypatch.context() as mp:
            for name in ("_group_norm_nchw", "_group_norm_rows", "add_channel_bias_"):
                real = getattr(pkg.ops, name)
                mp.setattr(pkg.ops, name, lambda *a, _real=real, _name=name, **k:
                           calls.append((_name, next(t for t in a if torch.is_tensor(t)).dtype)) or _real(*a, **k))
            with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
                inf_on = [o.float() for o in m.eval().forward_features(feats)[:2]]
        m.train()
        gen = torch.Generator(device=DEV).manual_seed(9)
        with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
            mask, low, multi = m.forward_features(feats)
        cots = [torch.randn(o.shape, device=DEV, generator=gen) for o in (mask, low, *multi)]
        got, got_g, fwd_on, bwd_on = _step(pkg, m, feats, cots, dtype)
        with monkeypatch.context() as mp:
            _refuse16(mp, pkg)
            with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
                inf_off = [o.float() for o in m.eval().forward_features(feats)[:2]]
            m.train()
            want, want_g, fwd_off, bwd_off = _step(pkg, m, feats, cots, dtype)
            moved, again_g, _, _ = _step(pkg, m, _perturbed(feats, dtype), cots, dtype)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.deterministic = flags
    out_err = max(_rel(a, b) for a, b in zip(got, want))
    out_spread = max(_rel(a, b) for a, b in zip(moved, want))
    inf_err = max(_rel(a, b) for a, b in zip(inf_on, inf_off))
    assert inf_err <= 3 * out_spread + 1e-5, (inf_err, out_spread)
    assert set(got_g) == set(want_g) and "input_proj.0.0.weight" in got_g and "feat::res2" in got_g
    err = {k: _rel(got_g[k], want_g[k]) for k in want_g}
    spread = {k: _rel(again_g[k], want_g[k]) for k in want_g}
    print(f"\n{dtype} decoder, 16-bit GroupNorm kernels against torch: outputs {out_err:.3g} (moved {out_spread:.3g}), "
          f"gradients {sorted(err.items(), key=lambda kv: -kv[1])[:3]}; moved features "
          f"{sorted(spread.items(), key=lambda kv: -kv[1])[:3]}")
    assert out_err <= 3 * out_spread + 1e-5, (out_err, out_spread)
    assert max(err.values()) <= 3 * max(spread.values()) + 1e-5, sorted(err.items(), key=lambda kv: -kv[1])[:4]
    assert all(dt == dtype for _, dt in calls), calls                   # every map the kernels took was 16-bit
    return sorted(name for name, _ in calls), fwd_on - fwd_off, bwd_on - bwd_off


@pytest.mark.parametrize("dtype", DTYPES)
def test_full_width_decoder_on_the_16bit_kernels(pkg, dtype, monkeypatch):
    """conv_dim 256: all five GroupNorms on the kernels (2 launches each forward; backward 3 per input projection,
    3 for the output convolution, 4 for the lateral), mask_features' bias in one pass in inference."""
    m, feats = _full_width_decoder(pkg)
    m = _autocast_twin(pkg, m, FULL_SHAPES, FULL_KW)
    inf, fwd, bwd = _on_and_off(pkg, m, feats, dtype, monkeypatch)
    assert fwd == 5 * 2 and bwd == 3 * 3 + 3 + 4
    assert inf == ["_group_norm_nchw"] * 2 + ["_group_norm_rows"] * 3 + ["add_channel_bias_"]


@pytest.mark.parametrize("dtype", DTYPES)
def test_golden_decoder_with_a_level_no_kernel_covers(pkg, dtype, monkeypatch):
    """The golden decoder's 2 x 3 stride-32 level: every input projection on its own (the NCHW kernel with fp32
    output where it covers the level, torch's GroupNorm on that one), the FPN maps on the 16-bit kernels."""
    m, feats, _ = build(pkg, device=DEV, fused=True, linear="tf32x3")
    torch.manual_seed(5)
    for proj in m.input_proj:
        torch.nn.init.normal_(proj[0].bias, std=0.1)
    m = _autocast_twin(pkg, m, PD_SHAPES, PD_KW)
    inf, fwd, bwd = _on_and_off(pkg, m, feats, dtype, monkeypatch)
    assert fwd == 4 * 2 and bwd == 3 * 2 + 3 + 4
    assert inf == ["_group_norm_nchw"] * 4 + ["add_channel_bias_"]


def decoder_steps_twice(dtype_name):
    """Two training steps of the full-width decoder under a 16-bit autocast (linear="autocast") with
    torch.use_deterministic_algorithms(True) and cudnn.deterministic -> "same" when outputs and gradients match."""
    from __graft_entry__ import load_package
    pkg = load_package()
    dtype = getattr(torch, dtype_name)
    m, feats = _full_width_decoder(pkg)
    m = _autocast_twin(pkg, m, FULL_SHAPES, FULL_KW).train()
    gen = torch.Generator(device=DEV).manual_seed(9)
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        shapes = [o.shape for o in (lambda r: (r[0], r[1], *r[2]))(m.forward_features(feats))]
    cots = [torch.randn(s, device=DEV, generator=gen) for s in shapes]
    torch.backends.cudnn.deterministic = True
    with deterministic_mode():
        (o1, g1, _, _), (o2, g2, _, _) = _step(pkg, m, feats, cots, dtype), _step(pkg, m, feats, cots, dtype)
    assert all(torch.equal(a, b) for a, b in zip(o1, o2))
    assert set(g1) == set(g2) and all(torch.equal(g1[n], g2[n]) for n in g1), [n for n in g1 if not torch.equal(g1[n], g2[n])]
    return "same"


@pytest.mark.parametrize("dtype", DTYPES)
def test_deterministic_decoder_training_steps(dtype):
    """In a fresh process whose environment sets CUBLAS_WORKSPACE_CONFIG from its start (as
    test_autocast_encoder_gpu.test_deterministic_training_steps does)."""
    code = (f"import sys; sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]\n"
            f"import test_group_norm_mixed_gpu as t\nprint(t.decoder_steps_twice({str(dtype).split('.')[-1]!r}))")
    env = dict(os.environ)
    env.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    args = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    res = subprocess.run(args, env=env, capture_output=True, text=True, timeout=1200)
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-4000:]
    assert res.stdout.strip().splitlines()[-1] == "same"


@pytest.mark.parametrize("dtype", DTYPES)
def test_linear_torch_under_autocast_runs_no_library_group_norm(pkg, dtype, monkeypatch):
    calls = []
    for name in ("_group_norm_nchw", "_group_norm_rows", "add_channel_bias_", "group_norm_backward",
                 "group_norm_rows_backward"):
        real = getattr(pkg.ops, name)
        monkeypatch.setattr(pkg.ops, name, lambda *a, _real=real, _name=name, **k: calls.append(_name) or _real(*a, **k))
    m, feats = _full_width_decoder(pkg)
    twin = pkg.pixel_decoder.MSDeformAttnPixelDecoder(FULL_SHAPES, fused=True, linear="torch", amp=True, **FULL_KW)
    twin.load_state_dict(m.state_dict())
    twin = twin.to(DEV).train()
    with torch.autocast("cuda", dtype=dtype):
        mask, low, multi = twin.forward_features(feats)
    (mask.float().sum() + low.float().sum() + sum(o.float().sum() for o in multi)).backward()
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        twin.eval().forward_features(feats)
    assert calls == []
