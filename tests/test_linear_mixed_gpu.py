"""The 16-bit Linear under torch.autocast (ops.linear_mixed, ops.linear_mixed_wgrad, LinearMixedFunction, and the
encoder's linear="autocast" path).

Contracts:
* forward / input gradient: every element within ulp16(y64) + 2^-16 * sum_k |x_k w_k| of the fp64 result on the same
  16-bit operands and fp32 bias (one rounding plus the fp32 accumulation); fp16 overflow gives +-inf; NaN / inf
  propagate like F.linear;
* weight / bias gradient: fp32, norm-relative error against fp64 no larger than torch's autocast weight gradient's,
  bit-identical from call to call;
* modules: every encoder Linear takes the new path under a 16-bit autocast (the input gradient on torch's GEMM
  except in deterministic mode, the inference forward where ops.linear_mixed_preferred says so), linear="torch"
  none of it, and the decoder stays within the one-ulp-perturbation bar of test_autocast_encoder_gpu against
  linear="torch".
"""
import pytest
import torch
import torch.nn.functional as F

from test_autocast_encoder_gpu import KW, _decoder, _features, _flat, _perturbed, _step, _weights
from test_mixed_precision_gpu import _nrel, _upcast_oracle_core, deterministic_mode

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DTYPES = [torch.bfloat16, torch.float16]
ERR_NULL, ERR_SHAPE, ERR_UNSUPPORTED = -1, -2, -3
WIDTHS = [96, 192, 256, 288, 1024]          # N and K of the full model's Linears
# (in, out) of the test decoders (d = 128 / 256, FFN 256 / 512, 4 heads) and tails of every kind
SMALL = [(128, 128), (128, 96), (128, 48), (128, 256), (256, 128), (256, 512), (512, 256), (8, 8), (40, 24)]


def ulp16(y, dtype):
    """One unit in the last place of the 16-bit type at |y| (float64 tensor)."""
    info = torch.finfo(dtype)
    mant = 7 if dtype == torch.bfloat16 else 10
    e = torch.floor(torch.log2(y.abs().clamp_min(info.smallest_normal)))
    return torch.exp2(e - mant)


def case(rows, k, n, dtype, seed=0, bias=True):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(rows, k, generator=gen).to(dtype).to(DEV)
    w = (torch.randn(n, k, generator=gen) / k ** 0.5).to(dtype).to(DEV)
    b = torch.randn(n, generator=gen).to(DEV) if bias else None
    return x, w, b


def check_bar(y, x, w, b, relu, dtype):
    y64 = x.double() @ w.double().t() + (b.double() if b is not None else 0.0)
    if relu:
        y64 = y64.clamp_min(0)
    bar = ulp16(y64, dtype) + 2.0 ** -16 * (x.double().abs() @ w.double().abs().t())
    err = (y.double() - y64).abs()
    assert y.dtype == dtype and y.shape == y64.shape
    assert bool((err <= bar).all()), f"max excess {(err - bar).max().item():.3e}"


# ---------------------------------------------------------------- 1./2. forward and input gradient
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("k", WIDTHS)
def test_forward_full_model_widths(pkg, dtype, k):
    for n in WIDTHS:
        for rows, bias, relu in ((300, True, False), (1, False, True), (257, True, True)):
            x, w, b = case(rows, k, n, dtype, seed=rows + n, bias=bias)
            check_bar(pkg.ops.linear_mixed(x, w, b, relu=relu), x, w, b, relu, dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("k,n", SMALL)
@pytest.mark.parametrize("rows", [1, 127, 128, 1000])
def test_forward_test_decoder_shapes_and_tails(pkg, dtype, k, n, rows):
    for bias, relu in ((True, False), (False, False), (True, True)):
        x, w, b = case(rows, k, n, dtype, seed=k * n + rows, bias=bias)
        check_bar(pkg.ops.linear_mixed(x, w, b, relu=relu), x, w, b, relu, dtype)


@pytest.mark.parametrize("dtype", DTYPES)
def test_forward_at_encoder_rows(pkg, dtype):
    x, w, b = case(172032, 256, 1024, dtype, seed=3)
    check_bar(pkg.ops.linear_mixed(x, w, b, relu=True), x, w, b, True, dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("k,n", [(256, 1024), (1024, 256), (288, 256), (96, 256)])
def test_input_gradient(pkg, dtype, k, n):
    """grad_x = grad_y @ w16: the forward kernel with the transposed weight, under the same bar."""
    gen = torch.Generator().manual_seed(k + n)
    g = torch.randn(3001, n, generator=gen).to(dtype).to(DEV)
    w = (torch.randn(n, k, generator=gen) / n ** 0.5).to(dtype).to(DEV)
    wt = w.t().contiguous()
    check_bar(pkg.ops.linear_mixed(g, wt), g, wt, None, False, dtype)


def test_fp16_overflow_is_inf(pkg):
    x = torch.full((130, 256), 100.0, dtype=torch.float16, device=DEV)
    w = torch.full((96, 256), 10.0, dtype=torch.float16, device=DEV)
    w[1] = -10.0
    y = pkg.ops.linear_mixed(x, w)
    assert torch.isinf(y[:, 0]).all() and (y[:, 0] > 0).all()
    assert torch.isinf(y[:, 1]).all() and (y[:, 1] < 0).all()


@pytest.mark.parametrize("dtype", DTYPES)
def test_non_finite_inputs_propagate_like_f_linear(pkg, dtype):
    x, w, b = case(300, 256, 192, dtype, seed=9)
    x[3, 7] = float("nan")
    x[10, 0] = float("inf")
    x[20, 5] = -float("inf")
    w[4, 9] = float("inf")
    for relu in (False, True):
        y = pkg.ops.linear_mixed(x, w, b, relu=relu).double()
        ref = F.linear(x.double(), w.double(), b.double())
        if relu:
            ref = F.relu(ref)
        assert torch.equal(y.isnan(), ref.isnan())
        assert torch.equal(y.isinf(), ref.isinf())
        inf = ref.isinf()
        assert torch.equal(y[inf], ref[inf])


# ---------------------------------------------------------------- 3. weight and bias gradient
def _wgrad64(g, x):
    return g.double().t() @ x.double(), g.double().sum(0)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("rows", [172032, 344064])
@pytest.mark.parametrize("out_f,in_f", [(256, 256), (1024, 256), (256, 1024), (288, 256)])
def test_wgrad_against_fp64_and_torch_autocast(pkg, dtype, rows, out_f, in_f):
    gen = torch.Generator().manual_seed(rows + out_f)
    g = (torch.randn(rows, out_f, generator=gen) * 1e-2).to(dtype).to(DEV)
    x = torch.randn(rows, in_f, generator=gen).to(dtype).to(DEV)
    gw, gb = pkg.ops.linear_mixed_wgrad(g, x)
    gw64, gb64 = _wgrad64(g, x)
    tw = (g.t() @ x).float()                          # torch's autocast weight gradient: a 16-bit GEMM result
    tb = g.sum(0).float()
    ours, theirs = _nrel(gw.double(), gw64), _nrel(tw.double(), gw64)
    ours_b, theirs_b = _nrel(gb.double(), gb64), _nrel(tb.double(), gb64)
    print(f"{dtype} rows={rows} {out_f}x{in_f}: grad_w nrel {ours:.3e} (torch autocast {theirs:.3e}), "
          f"grad_b nrel {ours_b:.3e} (torch {theirs_b:.3e})")
    assert gw.dtype == torch.float32 and gb.dtype == torch.float32
    assert ours <= theirs and ours_b <= theirs_b
    gw2, gb2 = pkg.ops.linear_mixed_wgrad(g, x)
    assert torch.equal(gw, gw2) and torch.equal(gb, gb2)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("rows", [1, 63, 1000, 20000])
@pytest.mark.parametrize("out_f,in_f", [(96, 256), (192, 288), (48, 128), (8, 40), (1024, 256), (256, 96)])
def test_wgrad_tails(pkg, dtype, rows, out_f, in_f):
    gen = torch.Generator().manual_seed(rows * 7 + out_f + in_f)
    g = torch.randn(rows, out_f, generator=gen).to(dtype).to(DEV)
    x = torch.randn(rows, in_f, generator=gen).to(dtype).to(DEV)
    for with_bias in (True, False):
        gw, gb = pkg.ops.linear_mixed_wgrad(g, x, with_bias=with_bias)
        gw64, gb64 = _wgrad64(g, x)
        bar = 2.0 ** -13 * (g.double().abs().t() @ x.double().abs())
        assert bool(((gw.double() - gw64).abs() <= bar).all())
        if with_bias:
            assert bool(((gb.double() - gb64).abs() <= 2.0 ** -13 * g.double().abs().sum(0)).all())
        else:
            assert gb is None


@pytest.mark.parametrize("dtype", DTYPES)
def test_wgrad_rows_split_across_images(pkg, dtype):
    """The images of a batch one call at a time, summed, against one call over all rows: within the bar."""
    gen = torch.Generator().manual_seed(5)
    g = torch.randn(4, 21504, 256, generator=gen).to(dtype).to(DEV)
    x = torch.randn(4, 21504, 256, generator=gen).to(dtype).to(DEV)
    gw, gb = pkg.ops.linear_mixed_wgrad(g.reshape(-1, 256), x.reshape(-1, 256))
    parts = [pkg.ops.linear_mixed_wgrad(g[i], x[i]) for i in range(4)]
    sw, sb = sum(p[0] for p in parts), sum(p[1] for p in parts)
    g2, x2 = g.reshape(-1, 256).double(), x.reshape(-1, 256).double()
    bar = 2.0 ** -13 * (g2.abs().t() @ x2.abs())
    assert bool(((gw.double() - sw.double()).abs() <= 2 * bar).all())
    assert bool(((gb.double() - sb.double()).abs() <= 2.0 ** -12 * g2.abs().sum(0)).all())


# ---------------------------------------------------------------- 4. LinearMixedFunction
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("relu,p", [(False, 0.0), (True, 0.0), (True, 0.25)])
@pytest.mark.parametrize("k,n", [(256, 1024), (1024, 256), (256, 288)])
def test_function_matches_autocast_composition(pkg, dtype, relu, p, k, n):
    gen = torch.Generator().manual_seed(k + n)
    x0 = torch.randn(2, 1500, k, generator=gen).to(dtype).to(DEV)
    lin = torch.nn.Linear(k, n).to(DEV)
    gy = torch.randn(2, 1500, n, generator=gen).to(dtype).to(DEV)

    def run(ours, mask=None):
        """mask: torch's composition with the ReLU replaced by our output's ReLU mask (for the gradients: where the
        two forwards round an output to opposite sides of zero, the ReLU keeps or drops a whole gradient element)."""
        lin.zero_grad(set_to_none=True)
        x = x0.clone().requires_grad_(True)
        torch.manual_seed(17)
        with torch.autocast("cuda", dtype=dtype):
            if ours:
                y = pkg.LinearMixedFunction.apply(x, lin.weight, lin.bias, relu, p)
            else:
                y = F.linear(x, lin.weight, lin.bias)
                if relu:
                    y = F.relu(y) if mask is None else y * mask
                y = F.dropout(y, p, training=True) if p else y
        y.backward(gy)
        return y.detach(), x.grad, lin.weight.grad.clone(), lin.bias.grad.clone()

    (y, gx, gw, gb), (ry, _, _, _) = run(True), run(False)
    _, rgx, rgw, rgb = run(False, (y > 0).to(dtype)) if relu else run(False)
    assert y.dtype == dtype and gx.dtype == dtype and gw.dtype == torch.float32 and gb.dtype == torch.float32
    if p:
        assert torch.equal(y == 0, ry == 0) or (y == 0).ne(ry == 0).float().mean() < 1e-3   # same mask, ReLU ties
    w16 = lin.weight.detach().to(dtype).double()
    sx = x0.reshape(-1, k).double().abs() @ w16.abs().t() / (1 - p) + lin.bias.detach().double().abs()
    assert bool(((y.reshape(-1, n).double() - ry.reshape(-1, n).double()).abs()
                 <= 2 * ulp16(ry.reshape(-1, n).double(), dtype) + 2.0 ** -15 * sx).all())
    for name, a, r in (("grad_x", gx, rgx), ("grad_w", gw, rgw), ("grad_b", gb, rgb)):
        e = _nrel(a.double(), r.double())
        print(f"{dtype} relu={relu} p={p} {k}->{n} {name}: nrel {e:.2e}")
        assert e <= 2.0 ** -8, name               # about one 16-bit rounding apart (torch rounds grad_w / grad_b)


def test_function_needs_input_grad(pkg):
    lin = torch.nn.Linear(256, 192).to(DEV)
    x = torch.randn(300, 256, device=DEV, dtype=torch.bfloat16)
    y = pkg.LinearMixedFunction.apply(x, lin.weight, lin.bias)
    y.float().sum().backward()
    assert lin.weight.grad is not None and lin.bias.grad is not None
    lin.zero_grad(set_to_none=True)
    lin.weight.requires_grad_(False)
    xg = x.clone().requires_grad_(True)
    pkg.LinearMixedFunction.apply(xg, lin.weight, lin.bias).float().sum().backward()
    assert lin.weight.grad is None and lin.bias.grad is not None and xg.grad is not None
    ref_b = torch.full((192,), 300.0, device=DEV)
    assert torch.equal(lin.bias.grad, ref_b)


# ---------------------------------------------------------------- 5. C ABI
@pytest.mark.parametrize("dtype", DTYPES)
def test_abi_errors(pkg, dtype):
    sfx = "bf16" if dtype == torch.bfloat16 else "f16"
    lib = pkg._lib.lib
    fwd, wg = getattr(lib, f"msda_b200_linear_mixed_{sfx}"), getattr(lib, f"msda_b200_linear_mixed_wgrad_{sfx}")
    x, w, b = case(200, 256, 96, dtype)
    y = torch.empty(200, 96, dtype=dtype, device=DEV)
    s = torch.cuda.current_stream().cuda_stream
    assert fwd(x.data_ptr(), w.data_ptr(), b.data_ptr(), y.data_ptr(), 200, 96, 256, 0, s) == 0
    assert fwd(None, w.data_ptr(), b.data_ptr(), y.data_ptr(), 200, 96, 256, 0, s) == ERR_NULL
    assert fwd(x.data_ptr(), None, b.data_ptr(), y.data_ptr(), 200, 96, 256, 0, s) == ERR_NULL
    assert fwd(x.data_ptr(), w.data_ptr(), b.data_ptr(), None, 200, 96, 256, 0, s) == ERR_NULL
    assert fwd(x.data_ptr(), w.data_ptr(), b.data_ptr(), y.data_ptr(), 0, 96, 256, 0, s) == ERR_SHAPE
    assert fwd(x.data_ptr() + 2, w.data_ptr(), b.data_ptr(), y.data_ptr(), 100, 96, 256, 0, s) == ERR_UNSUPPORTED
    assert fwd(x.data_ptr(), w.data_ptr(), b.data_ptr(), y.data_ptr(), 200, 96, 252, 0, s) == ERR_UNSUPPORTED
    assert fwd(x.data_ptr(), w.data_ptr(), b.data_ptr(), y.data_ptr(), 200, 92, 256, 0, s) == ERR_UNSUPPORTED
    gw = torch.empty(96, 256, device=DEV)
    nbytes = lib.msda_b200_linear_mixed_wgrad_workspace_bytes(200, 96, 256)
    assert nbytes > 0
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    args = [y.data_ptr(), x.data_ptr(), gw.data_ptr(), None, 200, 96, 256, ws.data_ptr(), s]
    assert wg(*args) == 0
    for i in (0, 1, 2, 7):
        bad = list(args)
        bad[i] = None
        assert wg(*bad) == ERR_NULL
    assert wg(*args[:4], 200, 0, 256, *args[7:]) == ERR_SHAPE
    assert wg(args[0] + 2, *args[1:]) == ERR_UNSUPPORTED
    assert wg(*args[:4], 200, 96, 252, *args[7:]) == ERR_UNSUPPORTED
    assert not pkg.ops.linear_mixed_supported(x[:, 2:], w[:, 2:])        # misaligned, non-contiguous view
    torch.cuda.synchronize()


# ---------------------------------------------------------------- 6. modules
def _records(pkg, monkeypatch):
    calls = []
    for name in ("linear_mixed", "linear_mixed_wgrad"):
        real = getattr(pkg.ops, name)
        monkeypatch.setattr(pkg.ops, name, lambda *a, _r=real, _n=name, **k: calls.append(_n) or _r(*a, **k))
    return calls


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("fused", [True, False])
def test_pixel_decoder_takes_the_new_path(pkg, oracle, monkeypatch, dtype, fused):
    feats = _features()
    m = _decoder(pkg, "autocast", fused=fused).train()
    ref = _decoder(pkg, "torch", fused=False, core=_upcast_oracle_core(oracle)).train()
    weights = _weights(ref, feats)
    layers = KW["transformer_enc_layers"]
    calls = _records(pkg, monkeypatch)
    outs, grads = _step(m, feats, dtype, weights)
    # six Linears per layer: forward on linear_mixed, weight gradient on linear_mixed_wgrad, input gradient on
    # torch's 16-bit GEMM (ops.linear_mixed_preferred)
    assert calls.count("linear_mixed_wgrad") == 6 * layers, calls
    assert calls.count("linear_mixed") == 6 * layers, calls
    del calls[:]
    ref_outs, ref_grads = _step(ref, feats, dtype, weights)
    assert not calls                                            # linear="torch" under autocast: none of it
    p_outs, p_grads = _step(ref, _perturbed(feats, dtype), dtype, weights)
    for i, (o, r, p) in enumerate(zip(outs, ref_outs, p_outs)):
        assert torch.isfinite(o).all()
        assert _nrel(o, r) <= _nrel(p, r), f"output {i}: {_nrel(o, r)} > {_nrel(p, r)}"
    for n in grads:
        assert torch.isfinite(grads[n]).all(), n
        assert _nrel(grads[n], ref_grads[n]) <= _nrel(p_grads[n], ref_grads[n]), n
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        del calls[:]
        got = [o.float() for o in _flat(m.eval().forward_features(feats))]
        n_inf = len(calls)
        want = [o.float() for o in _flat(ref.eval().forward_features(feats))]
        moved = [o.float() for o in _flat(ref.forward_features(_perturbed(feats, dtype)))]
    # folded position embedding (fused): stacked query GEMM + value + output + linear1 + linear2
    assert n_inf == (5 if fused else 6) * layers, calls
    for i, (o, r, p) in enumerate(zip(got, want, moved)):
        assert _nrel(o, r) <= _nrel(p, r), f"inference output {i}"


def _encoder(pkg, linear, fused):
    torch.manual_seed(0)
    return pkg.modules.MSDeformAttnTransformerEncoderOnly(d_model=256, nhead=8, num_encoder_layers=2,
                                                          dim_feedforward=1024, dropout=0.1, num_feature_levels=3,
                                                          enc_n_points=4, fused=fused, linear=linear).to(DEV)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("fused", [True, False])
def test_full_width_encoder(pkg, monkeypatch, dtype, fused):
    """d = 256, 8 heads, 3 levels, 4 points, FFN 1024 (dropout on in training): every Linear on the new kernels,
    forward and gradients within the one-ulp-perturbation bar of linear="torch"."""
    levels = [(32, 64), (16, 32), (8, 16)]
    gen = torch.Generator().manual_seed(1)
    srcs = [torch.randn(2, 256, h, w, generator=gen).to(DEV) for h, w in levels]
    pos = [torch.randn(2, 256, h, w, generator=gen).to(DEV) for h, w in levels]
    proj = torch.randn(2, sum(h * w for h, w in levels), 256, generator=gen).to(DEV)
    m, ref = _encoder(pkg, "autocast", fused).train(), _encoder(pkg, "torch", fused).train()
    calls = _records(pkg, monkeypatch)

    def step(mod, s):
        mod.zero_grad(set_to_none=True)
        torch.manual_seed(3)
        with torch.autocast("cuda", dtype=dtype):
            out = mod(s, pos)[0]
        (out.float() * proj).sum().backward()
        return out.detach().float(), {n: q.grad.float() for n, q in mod.named_parameters() if q.grad is not None}

    # dropout masks differ between the paths' generator use, so the bar is taken with dropout off
    for mod in (m, ref):
        for mm in mod.modules():
            if isinstance(mm, torch.nn.Dropout):
                mm.p = 0.0
    o, g = step(m, srcs)
    assert calls.count("linear_mixed_wgrad") == 12, calls
    del calls[:]
    r, rg = step(ref, srcs)
    assert not calls
    pert = [s + s.abs() * 2.0 ** -8 * torch.sign(torch.randn_like(s)) for s in srcs]
    p, pg = step(ref, pert)
    assert _nrel(o, r) <= _nrel(p, r)
    for n in g:
        assert _nrel(g[n], rg[n]) <= max(_nrel(pg[n], rg[n]), 1e-6), n
    # dropout on: the FFN's linear1 + ReLU + dropout is one node, still on the new kernels
    for mm in m.modules():
        if isinstance(mm, torch.nn.Dropout):
            mm.p = 0.1
    del calls[:]
    o2, g2 = step(m, srcs)
    assert calls.count("linear_mixed_wgrad") == 12 and torch.isfinite(o2).all()
    assert all(torch.isfinite(v).all() for v in g2.values())


_CUBLAS_NAMES = ("nvjet", "gemm", "cutlass", "xmma")


def _gemm_kernels(fn):
    """Names of the cuBLAS-style GEMM kernels that `fn` launches (torch.profiler, CUDA activity)."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                   and any(t in e.name.lower() for t in _CUBLAS_NAMES)})


@pytest.mark.parametrize("dtype", DTYPES)
def test_deterministic_training_runs_no_vendor_gemm(pkg, dtype):
    """With torch.use_deterministic_algorithms(True) every GEMM of the autocast encoder's training step is a library
    kernel (the input gradients too): no cuBLAS kernel in the trace, and two steps are bit-identical.  Without it the
    input gradients are torch's 16-bit GEMMs, where they are measured faster."""
    torch.manual_seed(0)
    m = _encoder(pkg, "autocast", True).train()
    levels = [(16, 32), (8, 16), (4, 8)]
    gen = torch.Generator().manual_seed(1)
    srcs = [torch.randn(2, 256, h, w, generator=gen).to(DEV) for h, w in levels]
    pos = [torch.randn(2, 256, h, w, generator=gen).to(DEV) for h, w in levels]
    proj = torch.randn(2, sum(h * w for h, w in levels), 256, generator=gen).to(DEV)
    out = {}

    def step():
        m.zero_grad(set_to_none=True)
        torch.manual_seed(5)
        with torch.autocast("cuda", dtype=dtype):
            o = m(srcs, pos)[0]
        (o.float() * proj).sum().backward()
        out["last"] = (o.detach().clone(), {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None})

    step()                                             # warm-up outside the trace
    with deterministic_mode():
        assert _gemm_kernels(step) == []
        o1, g1 = out["last"]
        step()
        o2, g2 = out["last"]
    assert torch.equal(o1, o2)
    assert set(g1) == set(g2) and all(torch.equal(g1[n], g2[n]) for n in g1)
    assert _gemm_kernels(step) != []                   # the input gradients on torch's GEMM


@pytest.mark.parametrize("dtype", DTYPES)
def test_shape_rules(pkg, monkeypatch, dtype):
    """Inference forward: torch's GEMM for 256 -> 256 without ReLU above 262 144 rows, the kernel at or below;
    input gradient: torch's GEMM, the kernel in deterministic mode."""
    lin = torch.nn.Linear(256, 256).to(DEV)
    calls = _records(pkg, monkeypatch)
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        for rows, want in ((262144, 1), (262145, 0)):
            del calls[:]
            x = torch.randn(rows, 256, device=DEV, dtype=dtype)
            y = pkg.modules._linear(lin, x, "autocast")
            assert y.dtype == dtype and calls.count("linear_mixed") == want, (rows, calls)
            check_bar(y[:4096], x[:4096], lin.weight.detach().to(dtype), lin.bias.detach(), False, dtype) \
                if want else None
    x = torch.randn(3000, 256, device=DEV, dtype=dtype, requires_grad=True)
    for det, want in ((False, 1), (True, 2)):
        del calls[:]
        with deterministic_mode() if det else torch.autograd.set_grad_enabled(True):
            pkg.LinearMixedFunction.apply(x, lin.weight, lin.bias).float().sum().backward()
        assert calls.count("linear_mixed") == want, (det, calls)


def test_weight_contract(pkg):
    """A non-contiguous weight is refused (torch's path), and a replaced weight is not served the old 16-bit copy."""
    lin = torch.nn.Linear(256, 256).to(DEV)
    x = torch.randn(300, 256, device=DEV, dtype=torch.bfloat16)
    assert not pkg.LinearMixedFunction.supported(x, lin.weight.t(), lin.bias)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        a = pkg.modules._linear(lin, x, "autocast")
        lin.weight = torch.nn.Parameter(lin.weight.detach() * 2)
        b = pkg.modules._linear(lin, x, "autocast")
    ref = F.linear(x.double(), (lin.weight.detach().to(torch.bfloat16)).double(), lin.bias.double())
    assert (b.double() - ref).abs().max().item() < (a.double() - ref).abs().max().item()
