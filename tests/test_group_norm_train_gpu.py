"""GPU tests of the GroupNorm training path: the training forwards and the backward kernels behind
GroupNormFunction / GroupNormRowsFunction, and the pixel decoder's training step on them.  Reference = torch
autograd of F.group_norm(x + cb) [-> relu] [+ F.interpolate(up)] in fp64 on the same fp32 inputs; the bar per
gradient is "no worse than torch's own fp32 autograd": err <= 2 * err32 + 1e-6 * max|ref|."""
import pytest
import torch
import torch.nn.functional as F

from test_pixel_decoder import build

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
EPS = 1e-5

# the seven cases of test_linear_gpu.py::test_group_norm_kernel_matches_torch, plus ReLU and up-sampling together
CASES = [
    ((2, 64, 12, 20), 32, False, None),
    ((2, 256, 16, 24), 32, True, None),
    ((3, 256, 24, 40), 32, False, (12, 20)),
    ((1, 64, 10, 28), 8, True, (7, 9)),
    ((2, 256, 96, 160), 32, False, (48, 80)),
    ((2, 64, 12, 39), 32, False, None),
    ((1, 256, 24, 78), 32, True, None),
    ((2, 128, 20, 36), 32, True, (10, 18)),
]


def _inputs(shape, groups, up, with_cb, seed):
    gen = torch.Generator().manual_seed(seed)
    N, C, H, W = shape
    x = torch.randn(shape, generator=gen) * 2.0 + 3.0                 # mean >> 0: the cancellation case
    w = torch.randn(C, generator=gen) * 0.3 + 1.0
    b = torch.randn(C, generator=gen) * 0.5
    cb = torch.randn(C, generator=gen) * 0.5 if with_cb else None
    u = torch.randn(N, C, *up, generator=gen) if up else None
    cot = torch.randn(shape, generator=gen)
    return [t.to(DEV) if t is not None else None for t in (x, w, b, cb, u, cot)]


def _torch_grads(tensors, groups, relu, cot, dtype):
    leaves = [t.detach().to(dtype).requires_grad_(True) if t is not None else None for t in tensors]
    x, w, b, cb, u = leaves
    z = x if cb is None else x + cb.view(1, -1, 1, 1)
    y = F.group_norm(z, groups, w, b, EPS)
    if relu:
        y = torch.relu(y)
    if u is not None:
        y = y + F.interpolate(u, size=x.shape[-2:], mode="bilinear", align_corners=False)
    (y * cot.to(dtype)).sum().backward()
    return [t.grad if t is not None else None for t in leaves]


def _assert_close_to_fp64(mine, tensors, groups, relu, cot):
    ref64 = _torch_grads(tensors, groups, relu, cot, torch.float64)
    ref32 = _torch_grads(tensors, groups, relu, cot, torch.float32)
    for name, g, r64, r32 in zip(("x", "weight", "bias", "channel_bias", "up"), mine, ref64, ref32):
        if r64 is None:
            assert g is None, name
            continue
        err = (g.double() - r64).abs().max().item()
        err32 = (r32.double() - r64).abs().max().item()
        assert err <= 2 * err32 + 1e-6 * r64.abs().max().item(), (name, err, err32)


@pytest.mark.parametrize("shape,groups,relu,up", CASES)
@pytest.mark.parametrize("with_cb", [False, True])
def test_group_norm_function_matches_fp64_autograd(pkg, shape, groups, relu, up, with_cb):
    x, w, b, cb, u, cot = _inputs(shape, groups, up, with_cb, seed=sum(shape) + groups)
    leaves = [t.clone().requires_grad_(True) if t is not None else None for t in (x, w, b, cb, u)]
    n0 = pkg.launch_count()
    y = pkg.GroupNormFunction.apply(*leaves, groups, EPS, relu)
    assert pkg.launch_count() - n0 == 2
    norm = torch.nn.GroupNorm(groups, shape[1], eps=EPS).to(DEV)
    with torch.no_grad():
        norm.weight.copy_(w)
        norm.bias.copy_(b)
        assert torch.equal(y, pkg.group_norm(x, norm, relu=relu, up=u, channel_bias=cb))
    n0 = pkg.launch_count()
    y.backward(cot)
    assert pkg.launch_count() - n0 == 3 + (u is not None)       # reduce, finalize, apply (+ the up-sampling adjoint)
    _assert_close_to_fp64([t.grad if t is not None else None for t in leaves], (x, w, b, cb, u), groups, relu, cot)
    # deterministic: the same bits on a second run
    _, mean_rstd = pkg.ops.group_norm_train(x, w, b, groups, EPS, relu=relu, up=u, channel_bias=cb)
    kw = dict(relu=relu, channel_bias=cb, up_shape=up, with_channel_bias=cb is not None)
    first = pkg.ops.group_norm_backward(cot, x, w, b, mean_rstd, groups, **kw)
    second = pkg.ops.group_norm_backward(cot, x, w, b, mean_rstd, groups, **kw)
    for g, t, r in zip(first, second, [t.grad if t is not None else None for t in leaves]):
        assert (g is None and t is None) or (torch.equal(g, t) and torch.equal(g, r))


def test_group_norm_function_honours_needs_input_grad(pkg):
    x, w, b, cb, u, cot = _inputs((2, 64, 8, 12), 32, (4, 6), True, seed=3)
    xl = x.clone().requires_grad_(True)
    y = pkg.GroupNormFunction.apply(xl, w, b, cb, u, 32, EPS, False)     # only x needs a gradient
    y.backward(cot)
    ref = _torch_grads((x, w, b, cb, u), 32, False, cot, torch.float64)[0]
    assert (xl.grad.double() - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()


LEVELS = [((2, 256, 8, 16), True), ((2, 256, 12, 39), True), ((2, 256, 24, 26), False)]   # W % 4 != 0 planes


def test_group_norm_rows_function_matches_fp64_autograd(pkg):
    """Three levels (KITTI-like planes with W % 4 != 0, one level without a convolution bias) as one node writing
    the concatenated [N, S, C] encoder input; the gradient arrives as a slice of a wider tensor."""
    groups = 32
    per_level = [_inputs(shape, groups, None, cb, seed=i + 11) for i, (shape, cb) in enumerate(LEVELS)]
    N, C = LEVELS[0][0][:2]
    sizes = [s[2] * s[3] for s, _ in LEVELS]
    S = sum(sizes)
    cot = torch.randn(N, S, C, device=DEV)
    leaves = [[t.clone().requires_grad_(True) if t is not None else None for t in p[:4]] for p in per_level]
    n0 = pkg.launch_count()
    out = pkg.GroupNormRowsFunction.apply(groups, EPS, *[t for lv in leaves for t in lv])
    assert pkg.launch_count() - n0 == 2 * len(LEVELS) and out.shape == (N, S, C)
    start = 0
    with torch.no_grad():
        for (x, w, b, cb, _, _), hw in zip(per_level, sizes):
            norm = torch.nn.GroupNorm(groups, C, eps=EPS).to(DEV)
            norm.weight.copy_(w)
            norm.bias.copy_(b)
            want = torch.empty(N, hw, C, device=DEV)
            pkg.ops.group_norm_rows(x, norm, want, channel_bias=cb)
            assert torch.equal(out[:, start:start + hw], want)
            start += hw
    # the gradient of the concatenated tensor as a slice of a wider one (the encoder's residual stream)
    wide = torch.zeros(N, S + 5, C, device=DEV)
    n0 = pkg.launch_count()
    (out * cot).sum().backward(inputs=[t for lv in leaves for t in lv if t is not None])
    assert pkg.launch_count() - n0 == 3 * len(LEVELS)
    start = 0
    for (x, w, b, cb, _, _), lv, hw, (shape, _) in zip(per_level, leaves, sizes, LEVELS):
        c = cot[:, start:start + hw].transpose(1, 2).reshape(shape)
        _assert_close_to_fp64([t.grad if t is not None else None for t in lv] + [None], (x, w, b, cb, None),
                              groups, False, c)
        start += hw
    # backward read straight from a strided slice: the same bits as from a contiguous copy
    x, w, b, cb = per_level[1][:4]
    dst = torch.full((N, S + 7, C), -7.0, device=DEV)
    rows = dst[:, 4:4 + sizes[1]]                                                    # a slice of a wider tensor
    mean_rstd = pkg.ops.group_norm_rows_train(x, w, b, groups, EPS, rows, channel_bias=cb)
    assert torch.equal(rows, out[:, sizes[0]:sizes[0] + sizes[1]].detach())
    assert bool((dst[:, :4] == -7.0).all()) and bool((dst[:, 4 + sizes[1]:] == -7.0).all())
    wide[:, 3:3 + sizes[1]] = cot[:, sizes[0]:sizes[0] + sizes[1]]
    a = pkg.ops.group_norm_rows_backward(wide[:, 3:3 + sizes[1]], x, w, b, mean_rstd, groups, channel_bias=cb,
                                         with_channel_bias=True)
    b2 = pkg.ops.group_norm_rows_backward(wide[:, 3:3 + sizes[1]].contiguous(), x, w, b, mean_rstd, groups,
                                          channel_bias=cb, with_channel_bias=True)
    for g, h in zip(a, b2):
        assert torch.equal(g, h)
    assert torch.equal(a[0], leaves[1][0].grad)


def test_group_norm_training_errors_and_fallback(pkg, monkeypatch):
    x, w, b, cb, u, cot = _inputs((1, 64, 6, 10), 32, (3, 5), False, seed=5)
    with pytest.raises(RuntimeError, match="group_norm_train needs"):
        pkg.ops.group_norm_train(x[..., :9].contiguous(), w, b, 32, EPS)           # H*W % 4 != 0
    with pytest.raises(RuntimeError, match="group_norm_train needs"):
        pkg.ops.group_norm_train(x, w[:-1], b, 32, EPS)
    y, mean_rstd = pkg.ops.group_norm_train(x, w, b, 32, EPS)
    with pytest.raises(RuntimeError, match="group_norm_backward needs"):
        pkg.ops.group_norm_backward(cot[..., :8].contiguous(), x, w, b, mean_rstd, 32)
    with pytest.raises(RuntimeError, match="mean_rstd must be"):
        pkg.ops.group_norm_backward(cot, x, w, b, mean_rstd[:, :16].contiguous(), 32)
    with pytest.raises(RuntimeError, match="group_norm_rows_backward needs"):
        pkg.ops.group_norm_rows_backward(torch.empty(1, 61, 64, device=DEV), x, w, b, mean_rstd, 32)
    # mis-aligned pointers pass the Python checks of the C ABI only when called directly: the library refuses them
    flat = torch.empty(x.numel() + 1, device=DEV)
    gx = flat[1:].view(x.shape)
    ws = torch.empty(int(pkg._lib.lib.msda_b200_group_norm_backward_workspace_bytes(1, 64)), dtype=torch.uint8,
                     device=DEV)
    rc = pkg._lib.lib.msda_b200_group_norm_backward_nchw_f32(
        cot.data_ptr(), x.data_ptr(), None, w.data_ptr(), b.data_ptr(), mean_rstd.data_ptr(), gx.data_ptr(),
        torch.empty_like(w).data_ptr(), torch.empty_like(b).data_ptr(), None, None, 1, 64, 6, 10, 32, 0, 0, 0,
        ws.data_ptr(), torch.cuda.current_stream().cuda_stream)
    with pytest.raises(RuntimeError, match="not supported|unsupported|UNSUPPORTED|code -3"):
        pkg._lib.check(rc, "group_norm_backward")
    # shapes the kernels do not cover take torch's path in the mirror, with no GroupNorm launch
    norm = torch.nn.GroupNorm(4, 8).to(DEV)
    conv = pkg.pixel_decoder._ConvNormAct(8, 8, kernel_size=1, norm=norm, activation=F.relu).to(DEV)
    xs = torch.randn(1, 8, 5, 7, device=DEV, requires_grad=True)
    n0 = pkg.launch_count()
    got = conv(xs, fused_norm=True)
    got.sum().backward()
    assert pkg.launch_count() - n0 == 0
    assert torch.allclose(got, torch.relu(norm(F.conv2d(xs, conv.weight, conv.bias))), atol=1e-6)


def _full_width_decoder(pkg):
    torch.manual_seed(5)
    kw = dict(transformer_dropout=0.0, transformer_nheads=8, transformer_dim_feedforward=1024,
              transformer_enc_layers=2, conv_dim=256, mask_dim=256, norm="GN",
              transformer_in_features=["res3", "res4", "res5"], common_stride=4)
    shapes = {"res2": (96, 4), "res3": (192, 8), "res4": (384, 16), "res5": (768, 32)}
    m = pkg.pixel_decoder.MSDeformAttnPixelDecoder(shapes, fused=True, linear="tf32x3", **kw).cuda().train()
    for mod in m.modules():                                    # away from the zero-initialised producers
        if isinstance(mod, pkg.modules.MSDeformAttn):
            torch.nn.init.normal_(mod.sampling_offsets.weight, std=0.02)
            torch.nn.init.normal_(mod.attention_weights.weight, std=0.05)
    for proj in m.input_proj:                                  # a non-zero convolution bias, so that it gets tested
        torch.nn.init.normal_(proj[0].bias, std=0.1)
    feats = {k: torch.randn(2, c, 128 // s, 256 // s, device="cuda:0") for k, (c, s) in shapes.items()}
    return m, feats


def _train_step(pkg, m, feats, cots):
    leaves = {k: v.clone().requires_grad_(True) for k, v in feats.items()}
    m.zero_grad(set_to_none=True)
    n0 = pkg.launch_count()
    mask, low, multi = m.forward_features(leaves)
    fwd = pkg.launch_count() - n0
    outs = [mask, low, *multi]
    loss = sum((o * c).sum() for o, c in zip(outs, cots))
    n0 = pkg.launch_count()
    loss.backward()
    bwd = pkg.launch_count() - n0
    grads = {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}
    grads.update({"feat::" + k: v.grad.clone() for k, v in leaves.items()})
    return [o.detach() for o in outs], grads, fwd, bwd


def _steps_with_the_kernels_on_and_off(pkg, m, feats, monkeypatch):
    """One forward_features + backward with the GroupNorm kernels on, the same step with them off (both predicates
    patched to False: torch's path), and that torch step on features moved by ~1e-6.  -> (forward launches on - off,
    backward launches on - off, worst output error, per-tensor gradient error, per-tensor spread of the moved step)."""
    flags = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.deterministic)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.deterministic = True
    try:
        with torch.no_grad():
            mask, low, multi = m.forward_features(feats)
            shapes = [mask.shape, low.shape, *[o.shape for o in multi]]
        gen = torch.Generator(device="cuda:0").manual_seed(9)
        cots = [torch.randn(s, device="cuda:0", generator=gen) for s in shapes]
        got, got_g, fwd_on, bwd_on = _train_step(pkg, m, feats, cots)
        with monkeypatch.context() as mp:
            mp.setattr(pkg.ops, "group_norm_supported", lambda *a, **k: False)
            mp.setattr(pkg.ops, "group_norm_rows_supported", lambda *a, **k: False)
            want, want_g, fwd_off, bwd_off = _train_step(pkg, m, feats, cots)
            # the torch path on features moved by ~1e-6: a forward that differs as much as the kernels' does.  The
            # decoder's gradients are discontinuous in its forward values (ReLU masks, the bilinear cells of the
            # deformable sampling), so this, not a rerun on identical inputs, is the spread to expect
            gen = torch.Generator(device="cuda:0").manual_seed(10)
            moved = {k: v + 1e-6 * torch.randn(v.shape, device="cuda:0", generator=gen) for k, v in feats.items()}
            _, again_g, _, _ = _train_step(pkg, m, moved, cots)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.deterministic = flags
    worst_out = 0.0
    for a, b in zip(got, want):
        worst_out = max(worst_out, (a - b).abs().max().item() / max(1e-30, b.abs().max().item()))
    assert set(got_g) == set(want_g) and "input_proj.0.0.bias" in got_g and "feat::res2" in got_g

    def rel(a, b):                      # per tensor: |a - b| / |b| (Frobenius norms)
        return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()
    err = {k: rel(got_g[k], want_g[k]) for k in want_g}
    spread = {k: rel(again_g[k], want_g[k]) for k in want_g}
    top = sorted(err.items(), key=lambda kv: -kv[1])[:4]
    print(f"\ndecoder training step, GroupNorm kernels against torch: outputs {worst_out:.3g}, gradients {top}; "
          f"torch against torch on moved features: {sorted(spread.items(), key=lambda kv: -kv[1])[:4]}")
    return fwd_on - fwd_off, bwd_on - bwd_off, worst_out, err, spread


def test_decoder_training_step_on_the_group_norm_kernels_matches_the_torch_path(pkg, monkeypatch):
    """One forward_features + backward of the full-width decoder with the GroupNorm kernels on against the same step
    with them off (today's torch path): outputs, every parameter gradient and the feature gradients agree."""
    m, feats = _full_width_decoder(pkg)
    fwd, bwd, worst_out, err, spread = _steps_with_the_kernels_on_and_off(pkg, m, feats, monkeypatch)
    # five GroupNorms: 2 launches each forward; backward 3 per input projection, 3 for the output convolution and
    # 4 for the lateral (its up-sampled add)
    assert fwd == 5 * 2 and bwd == 3 * 3 + 3 + 4
    assert worst_out <= 1e-4, worst_out
    # observed on a B200: outputs 6.0e-07; gradients at most 1.5e-3 (layers.0.linear1.weight), torch on the moved
    # features at most 1.4e-3 (adapter_1.norm.weight); torch rerun on identical inputs 5e-7
    assert max(err.values()) <= 3 * max(spread.values()) + 1e-5, sorted(err.items(), key=lambda kv: -kv[1])[:4]


def test_decoder_training_step_with_a_level_the_kernels_do_not_cover(pkg, monkeypatch):
    """The golden decoder's pyramid has a stride-32 level of 2 x 3 pixels, which no GroupNorm kernel covers: in
    training too, the covered maps (the stride-8 and stride-16 input projections, the lateral and the output
    convolution) run on the kernels and that level on torch's path, each input projection on its own."""
    m, feats, _ = build(pkg, device="cuda:0", fused=True, linear="tf32x3")
    m.train()
    torch.manual_seed(5)
    for proj in m.input_proj:                                  # a non-zero convolution bias, so that it gets tested
        torch.nn.init.normal_(proj[0].bias, std=0.1)
    fwd, bwd, worst_out, err, spread = _steps_with_the_kernels_on_and_off(pkg, m, feats, monkeypatch)
    assert fwd == 4 * 2 and bwd == 3 * 2 + 3 + 4
    assert worst_out <= 1e-4, worst_out
    assert max(err.values()) <= 3 * max(spread.values()) + 1e-5, sorted(err.items(), key=lambda kv: -kv[1])[:4]
