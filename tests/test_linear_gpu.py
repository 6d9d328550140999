"""GPU tests of msda_b200_linear_f32 (SURVEY.md 8f.3): the fp32 nn.Linear of the layers around the op
(ops/modules/ms_deform_attn.py:62-65, msdeformattn.py:126-130) as an error-compensated 3xTF32 GEMM on the
tensor cores.  Reference = torch.nn.functional.linear in fp64; the bar is "as accurate as an fp32 GEMM":
the error against fp64 may not exceed a small multiple of the error torch's own fp32 (non-TF32) GEMM makes
on the same inputs."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
# measured: 1.0-1.6x.  The tensor core truncates when it adds into the fp32 accumulator, so the error grows
# with the number of accumulations per accumulator: in_features >= 512 use four accumulators (1.3x at 1024;
# with two it was 2.9x)
ERR_FACTOR = 3.0


def case(rows, out_f, in_f, seed, bias=True, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(rows, in_f, generator=g) * scale).to(DEV)
    w = (torch.randn(out_f, in_f, generator=g) / in_f ** 0.5).to(DEV)
    b = torch.randn(out_f, generator=g).to(DEV) if bias else None
    return x, w, b


@pytest.mark.parametrize("rows,out_f,in_f", [
    (128, 256, 32), (128, 256, 256), (1, 256, 256), (127, 256, 256), (129, 256, 256), (1000, 192, 256),
    (777, 96, 256), (513, 1024, 256), (640, 256, 1024), (130, 128, 64), (300, 64, 96), (50, 4, 32),
    (260, 260, 64), (333, 512, 128)])
def test_linear_matches_fp64(pkg, rows, out_f, in_f):
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        x, w, b = case(rows, out_f, in_f, seed=rows + out_f)
        n0 = pkg.launch_count()
        y = pkg.linear_tf32x3(x, w, b)
        torch.cuda.synchronize()
        assert pkg.launch_count() - n0 == 2           # weight split + GEMM
        ref64 = F.linear(x.double(), w.double(), b.double())
        err = (y.double() - ref64).abs().max().item()
        err32 = (F.linear(x, w, b).double() - ref64).abs().max().item()
        assert y.shape == (rows, out_f) and torch.isfinite(y).all()
        assert err <= ERR_FACTOR * err32 + 1e-7, (err, err32)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def test_linear_is_far_more_accurate_than_plain_tf32(pkg):
    x, w, b = case(512, 256, 256, seed=5)
    ref64 = F.linear(x.double(), w.double(), b.double())
    err = (pkg.linear_tf32x3(x, w, b).double() - ref64).abs().max().item()
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        err_tf32 = (F.linear(x, w, b).double() - ref64).abs().max().item()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    assert err * 50 < err_tf32, (err, err_tf32)


def test_linear_relu_no_bias_leading_dims_and_scales(pkg):
    x, w, b = case(2 * 77, 192, 256, seed=9)
    x3 = x.view(2, 77, 256)
    y = pkg.linear_tf32x3(x3, w, None, relu=True)
    assert y.shape == (2, 77, 192)
    ref = F.linear(x3.double(), w.double()).relu()
    assert (y.double() - ref).abs().max().item() <= 2e-5
    assert (y >= 0).all()
    # large / small magnitudes: relative accuracy is what the split preserves
    for scale in (1e-6, 1e4):
        xs, ws, bs = case(256, 256, 256, seed=3, bias=False, scale=scale)
        ys = pkg.linear_tf32x3(xs, ws, None)
        refs = F.linear(xs.double(), ws.double())
        assert (ys.double() - refs).abs().max().item() <= 3e-6 * refs.abs().max().item()
    # exactly representable inputs give the exact result (integers: no rounding anywhere)
    xi = torch.randint(-8, 9, (200, 64), device=DEV).float()
    wi = torch.randint(-8, 9, (32, 64), device=DEV).float()
    assert torch.equal(pkg.linear_tf32x3(xi, wi, None), F.linear(xi.double(), wi.double()).float())


def test_linear_non_finite_inputs_propagate(pkg):
    x, w, b = case(130, 64, 64, seed=2)
    x[5, 7] = float("inf")
    x[100, 0] = float("nan")
    y = pkg.linear_tf32x3(x, w, b)
    assert not torch.isfinite(y[5]).any() and torch.isnan(y[100]).all()
    keep = torch.ones(130, dtype=torch.bool, device=DEV)
    keep[5] = keep[100] = False
    assert torch.isfinite(y[keep]).all()


def test_linear_error_behaviour(pkg):
    x, w, b = case(64, 64, 64, seed=1)
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        pkg.linear_tf32x3(x.cpu(), w.cpu(), b.cpu())
    with pytest.raises(RuntimeError, match="contiguous"):
        pkg.linear_tf32x3(x.t(), w, b)
    with pytest.raises(RuntimeError, match="float32"):
        pkg.linear_tf32x3(x.double(), w.double(), b.double())
    with pytest.raises(RuntimeError, match="in % 32"):
        pkg.linear_tf32x3(x[:, :48].contiguous(), w[:, :48].contiguous(), b)
    # the C ABI itself: null pointers and unsupported shapes are reported, nothing is launched
    lib = pkg._lib.lib
    assert lib.msda_b200_linear_f32(None, w.data_ptr(), None, x.data_ptr(), 64, 64, 64, 0, x.data_ptr(), None) == -1
    assert lib.msda_b200_linear_f32(x.data_ptr(), w.data_ptr(), None, x.data_ptr(), 64, 64, 48, 0, x.data_ptr(), None) == -3
    assert lib.msda_b200_linear_f32(x.data_ptr(), w.data_ptr(), None, x.data_ptr(), 0, 64, 64, 0, x.data_ptr(), None) == -2


def test_encoder_layer_with_tensor_core_linears_matches_torch_linears(pkg):
    """The encoder mirror with linear="tf32x3" (inference) against the same weights with torch's fp32
    GEMMs; with autograd on it must take the torch path (and be bit-identical to it)."""
    torch.manual_seed(4)
    levels = [(8, 16), (16, 32), (32, 64)]
    kw = dict(d_model=256, nhead=8, num_encoder_layers=2, dim_feedforward=1024, dropout=0.0,
              num_feature_levels=3, enc_n_points=4)
    a = pkg.modules.MSDeformAttnTransformerEncoderOnly(**kw).to(DEV).eval()
    b = pkg.modules.MSDeformAttnTransformerEncoderOnly(linear="tf32x3", **kw).to(DEV).eval()
    b.load_state_dict(a.state_dict())
    for m in list(a.modules()) + list(b.modules()):           # away from the zero-initialised producers
        if isinstance(m, pkg.modules.MSDeformAttn):
            torch.nn.init.normal_(m.sampling_offsets.weight, std=0.02)
            torch.nn.init.normal_(m.attention_weights.weight, std=0.05)
    b.load_state_dict(a.state_dict())
    srcs = [torch.randn(2, 256, h, w, device=DEV) for h, w in levels]
    pos = [torch.randn(2, 256, h, w, device=DEV) for h, w in levels]
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            n0 = pkg.launch_count()
            ya = a(srcs, pos)[0]
            n1 = pkg.launch_count()
            yb = b(srcs, pos)[0]
            n2 = pkg.launch_count()
        assert n1 - n0 == 2 and n2 - n1 == 2 + (2 * 6 + 2) * 2   # + ((split + GEMM) x 6 linears + 2 add-norms) x 2 layers
        assert (ya - yb).abs().max().item() <= 5e-5, (ya - yb).abs().max().item()
        # autograd on: forward and grad_x GEMMs on the tensor cores, everything else torch
        srcs_a = [t.clone().requires_grad_(True) for t in srcs]
        srcs_b = [t.clone().requires_grad_(True) for t in srcs]
        cot = torch.randn_like(ya)
        (a(srcs_a, pos)[0] * cot).sum().backward()
        n3 = pkg.launch_count()
        yc = b(srcs_b, pos)[0]
        (yc * cot).sum().backward()
        # per layer: MSDA fwd + bwd, 6 x (split + GEMM) forward, 6 x (split + GEMM) for grad_x,
        # 6 weight / bias gradient kernels, 2 x (add + LayerNorm forward, backward)
        assert pkg.launch_count() - n3 == 2 * (3 + 12 + 12 + 6 + 4)   # MSDA backward = 2 gated kernels
        assert (yc - ya).abs().max().item() <= 5e-5
        # gradients pass through floor() of the sampling locations: a 1e-6 difference in a location next to
        # a cell edge moves the point into the neighbouring cell, where the location gradient differs by
        # O(1).  torch against torch with 1e-6 input noise differs by 4e-4 .. 5e-3 in relative L2 here
        # (measured), so that is the yardstick; everything downstream of the last MSDA
        # call (last layer's FFN) has no such term and must agree to rounding
        def rel(u, v):
            return (u - v).norm().item() / max(v.norm().item(), 1e-12)
        for ga, gb in zip(srcs_a, srcs_b):
            assert rel(gb.grad, ga.grad) <= 1e-2
        last = f"encoder.layers.{kw['num_encoder_layers'] - 1}."
        for (na, pa), (nb, pb) in zip(a.named_parameters(), b.named_parameters()):
            if pa.grad is not None:
                exact = na.startswith(last) and ("linear2" in na or "norm2" in na)
                assert rel(pb.grad, pa.grad) <= (2e-5 if exact else 1e-2), na
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


@pytest.mark.parametrize("rows,cols,with_res", [(1000, 256, True), (37, 256, False), (513, 128, True),
                                                (64, 512, True), (9, 384, True)])
def test_add_layernorm_matches_torch(pkg, rows, cols, with_res):
    g = torch.Generator().manual_seed(rows)
    x = (torch.randn(rows, cols, generator=g) * 3 + 1).to(DEV)
    r = torch.randn(rows, cols, generator=g).to(DEV) if with_res else None
    w = torch.randn(cols, generator=g).to(DEV)
    b = torch.randn(cols, generator=g).to(DEV)
    y = pkg.add_layernorm(x, r, w, b, 1e-5)
    v = x.double() + (r.double() if with_res else 0)
    ref = F.layer_norm(v, (cols,), w.double(), b.double(), 1e-5)
    ref32 = F.layer_norm(x + r if with_res else x, (cols,), w, b, 1e-5)
    err, err32 = (y.double() - ref).abs().max().item(), (ref32.double() - ref).abs().max().item()
    assert err <= 2 * err32 + 1e-6, (err, err32)
    with pytest.raises(RuntimeError, match="add_layernorm needs"):
        pkg.add_layernorm(x[:, :100].contiguous(), None, w[:100].contiguous(), b[:100].contiguous())


def test_linear_autograd_function_matches_torch(pkg):
    x, w, b = case(500, 256, 128, seed=12)
    x1, w1, b1 = (t.clone().requires_grad_(True) for t in (x, w, b))
    x2, w2, b2 = (t.clone().requires_grad_(True) for t in (x, w, b))
    cot = torch.randn(500, 256, device=DEV)
    (pkg.LinearTF32x3Function.apply(x1, w1, b1) * cot).sum().backward()
    (F.linear(x2.double(), w2.double(), b2.double()) * cot.double()).sum().backward()
    for mine, ref in ((x1, x2), (w1, w2), (b1, b2)):
        assert (mine.grad.double() - ref.grad.double()).abs().max().item() <= 1e-5 * max(1.0, ref.grad.abs().max().item())


def test_linear_autograd_function_with_relu_in_the_epilogue(pkg):
    """apply(x, w, b, True) == F.relu(F.linear(x, w, b)) forward and backward (the mask comes from the saved output)."""
    x, w, b = case(700, 1024, 256, seed=13)
    x1, w1, b1 = (t.clone().requires_grad_(True) for t in (x, w, b))
    x2, w2, b2 = (t.clone().requires_grad_(True) for t in (x, w, b))
    cot = torch.randn(700, 1024, device=DEV)
    n0 = pkg.launch_count()
    y1 = pkg.LinearTF32x3Function.apply(x1, w1, b1, True)
    assert pkg.launch_count() - n0 == 2 and float(y1.detach().min()) == 0.0
    (y1 * cot).sum().backward()
    y2 = F.relu(F.linear(x2.double(), w2.double(), b2.double()))
    # the sign of an output within rounding of zero may differ between the two GEMMs: mask the cotangent there
    near_zero = (F.linear(x.double(), w.double(), b.double()).abs() < 1e-5)
    assert (y1.double() - y2).abs().max().item() <= 1e-5
    (y2 * cot.double().masked_fill(near_zero, 0.0)).sum().backward()
    x3, w3, b3 = (t.clone().requires_grad_(True) for t in (x, w, b))
    (pkg.LinearTF32x3Function.apply(x3, w3, b3, True) * cot.masked_fill(near_zero, 0.0)).sum().backward()
    for mine, ref in ((x3, x2), (w3, w2), (b3, b2)):
        assert (mine.grad.double() - ref.grad.double()).abs().max().item() <= 2e-5 * max(1.0, ref.grad.abs().max().item())


def test_linear_autograd_function_with_relu_and_dropout(pkg):
    """apply(x, w, b, True, p) == F.dropout(F.relu(F.linear(x, w, b)), p, True) with the same generator state: the
    same mask (torch's own dropout kernel draws it), the same outputs and gradients."""
    x, w, b = case(600, 1024, 256, seed=14)
    p = 0.1
    cot = torch.randn(600, 1024, device=DEV)
    near_zero = (F.linear(x.double(), w.double(), b.double()).abs() < 1e-5)
    cot = cot.masked_fill(near_zero, 0.0)
    x1, w1, b1 = (t.clone().requires_grad_(True) for t in (x, w, b))
    x2, w2, b2 = (t.clone().requires_grad_(True) for t in (x, w, b))
    torch.manual_seed(99)
    y1 = pkg.LinearTF32x3Function.apply(x1, w1, b1, True, p)
    (y1 * cot).sum().backward()
    torch.manual_seed(99)
    y2 = F.dropout(F.relu(F.linear(x2.double(), w2.double(), b2.double())).float(), p, True)
    dropped = (y2 == 0) & (F.linear(x.double(), w.double(), b.double()) > 1e-5)
    assert 0.05 < dropped.float().mean().item() / max((F.linear(x.double(), w.double(), b.double()) > 1e-5).float().mean().item(), 1e-9) < 0.15
    assert torch.equal((y1 == 0) | near_zero, (y2 == 0) | near_zero)          # the same mask
    assert (y1.double() - y2.double()).abs().max().item() <= 2e-5
    (y2.double() * cot.double()).sum().backward()
    for mine, ref in ((x1, x2), (w1, w2), (b1, b2)):
        assert (mine.grad.double() - ref.grad.double()).abs().max().item() <= 2e-5 * max(1.0, ref.grad.abs().max().item())
    with pytest.raises(ValueError, match="dropout_p needs"):
        pkg.LinearTF32x3Function.apply(x1, w1, b1, False, p)


@pytest.mark.parametrize("rows,out_f,in_f", [(4096, 256, 256), (8192, 96, 256), (2080, 1024, 256), (6400, 256, 1024),
                                            (64, 128, 64)])
def test_linear_weight_gradient_gemm_split_k_in_kernel_split(pkg, rows, out_f, in_f):
    """grad_w = grad_y^T @ x through the same kernel: transposed operands, 'weight' split in the kernel,
    reduction over the rows spread over several CTAs per output tile (reductions into a zeroed output)."""
    g = torch.Generator().manual_seed(rows + in_f)
    gy = torch.randn(rows, out_f, generator=g).to(DEV)
    x = torch.randn(rows, in_f, generator=g).to(DEV)
    gyt, xt = pkg.ops.transpose2d(gy), pkg.ops.transpose2d(x)
    assert torch.equal(gyt, gy.t().contiguous()) and torch.equal(xt, x.t().contiguous())
    gw = pkg.linear_tf32x3(gyt, xt, None, split_weight_in_kernel=True)
    ref = gy.double().t() @ x.double()
    err = (gw.double() - ref).abs().max().item()
    err32 = ((gy.t() @ x).double() - ref).abs().max().item()
    assert gw.shape == (out_f, in_f)
    assert err <= ERR_FACTOR * err32 + 1e-6, (err, err32)


def test_transpose2d_ragged_shapes(pkg):
    for rows, cols in ((1, 1), (33, 7), (100, 257), (1000, 96)):
        x = torch.randn(rows, cols, device=DEV)
        assert torch.equal(pkg.ops.transpose2d(x), x.t().contiguous())
    with pytest.raises(RuntimeError, match="transpose2d needs"):
        pkg.ops.transpose2d(torch.randn(4, 4, device=DEV).t())


def test_linear_full_size_is_exact_on_integer_inputs(pkg):
    """BASELINE configs[2] row count (1024x2048 pyramid, batch 8 = 344 064 rows): thousands of tiles per
    persistent CTA, every barrier phase flips many times.  Small-integer inputs make every product and sum
    exactly representable, so the result must equal the fp64 one bit for bit, for every tile."""
    g = torch.Generator().manual_seed(7)
    rows = 344064
    for out_f, in_f in ((256, 256), (96, 256), (256, 1024)):
        x = torch.randint(-4, 5, (rows, in_f), generator=g).float().to(DEV)
        w = torch.randint(-4, 5, (out_f, in_f), generator=g).float().to(DEV)
        b = torch.randint(-9, 10, (out_f,), generator=g).float().to(DEV)
        y = pkg.linear_tf32x3(x, w, b)
        ref = (x.double() @ w.double().t() + b.double()).float()
        assert torch.equal(y, ref), (out_f, in_f, (y - ref).abs().max().item())
        del x, w, y, ref
    # weight-gradient shape at the training row count: split-K, reductions into the zeroed output
    rows = 172032
    gy = torch.randint(-2, 3, (rows, 192), generator=g).float().to(DEV)
    x = torch.randint(-2, 3, (rows, 256), generator=g).float().to(DEV)
    gw = pkg.linear_tf32x3(pkg.ops.transpose2d(gy), pkg.ops.transpose2d(x), None, split_weight_in_kernel=True)
    assert torch.equal(gw, (gy.double().t() @ x.double()).float())
    gw2, gb2 = pkg.ops.linear_wgrad(gy, x)
    assert torch.equal(gw2, gw) and torch.equal(gb2, gy.double().sum(0).float())


def test_add_layernorm_full_size(pkg):
    g = torch.Generator().manual_seed(8)
    x = torch.randn(344064, 256, generator=g).to(DEV)
    r = torch.randn(344064, 256, generator=g).to(DEV)
    w = torch.randn(256, generator=g).to(DEV)
    b = torch.randn(256, generator=g).to(DEV)
    y = pkg.add_layernorm(x, r, w, b, 1e-5)
    ref = F.layer_norm(x + r, (256,), w, b, 1e-5)
    assert (y - ref).abs().max().item() <= 5e-6


@pytest.mark.parametrize("rows,out_f,in_f", [(4096, 256, 256), (8200, 96, 256), (2085, 1024, 256), (6400, 256, 1024),
                                            (33, 128, 64), (1000, 100, 36), (5, 4, 4)])
def test_linear_wgrad_kernel(pkg, rows, out_f, in_f):
    """grad_W = grad_y^T @ x and grad_b = column sums, reduction over the rows, operands not transposed in
    memory (A through tensor memory, B re-laid out in shared memory), against fp64 and torch's fp32 kernels."""
    g = torch.Generator().manual_seed(rows + in_f)
    gy = torch.randn(rows, out_f, generator=g).to(DEV)
    x = torch.randn(rows, in_f, generator=g).to(DEV)
    gw, gb = pkg.ops.linear_wgrad(gy, x)
    ref = gy.double().t() @ x.double()
    err, err32 = (gw.double() - ref).abs().max().item(), ((gy.t() @ x).double() - ref).abs().max().item()
    assert gw.shape == (out_f, in_f) and err <= ERR_FACTOR * err32 + 2e-6 * ref.abs().max().item(), (err, err32)
    refb = gy.double().sum(0)
    assert (gb.double() - refb).abs().max().item() <= 4 * (gy.sum(0).double() - refb).abs().max().item() + 1e-4
    gw2, none = pkg.ops.linear_wgrad(gy, x, with_bias=False)
    assert none is None and (gw2 - gw).abs().max().item() <= 2e-3 * max(1.0, gw.abs().max().item())
    # exact on small integers, at every tile / chunk boundary
    gyi = torch.randint(-2, 3, (rows, out_f), generator=g).float().to(DEV)
    xi = torch.randint(-2, 3, (rows, in_f), generator=g).float().to(DEV)
    gwi, gbi = pkg.ops.linear_wgrad(gyi, xi)
    assert torch.equal(gwi, (gyi.double().t() @ xi.double()).float())
    assert torch.equal(gbi, gyi.double().sum(0).float())
    with pytest.raises(RuntimeError, match="linear_wgrad needs"):
        pkg.ops.linear_wgrad(gy[:, :out_f - 1].contiguous(), x)


@pytest.mark.parametrize("rows,cols", [(1000, 256), (77, 128), (20000, 256)])
def test_add_layernorm_autograd_function(pkg, rows, cols):
    g = torch.Generator().manual_seed(rows)
    x = (torch.randn(rows, cols, generator=g) * 2 + 0.5).to(DEV)
    r = torch.randn(rows, cols, generator=g).to(DEV)
    w = (torch.randn(cols, generator=g) + 1).to(DEV)
    b = torch.randn(cols, generator=g).to(DEV)
    cot = torch.randn(rows, cols, generator=g).to(DEV)
    leaves = [t.clone().requires_grad_(True) for t in (x, r, w, b)]
    (pkg.AddLayerNormFunction.apply(*leaves, 1e-5) * cot).sum().backward()
    ref = [t.clone().double().requires_grad_(True) for t in (x, r, w, b)]
    (F.layer_norm(ref[0] + ref[1], (cols,), ref[2], ref[3], 1e-5) * cot.double()).sum().backward()
    t32 = [t.clone().requires_grad_(True) for t in (x, r, w, b)]
    (F.layer_norm(t32[0] + t32[1], (cols,), t32[2], t32[3], 1e-5) * cot).sum().backward()
    for mine, r64, r32 in zip(leaves, ref, t32):
        err = (mine.grad.double() - r64.grad).abs().max().item()
        err32 = (r32.grad.double() - r64.grad).abs().max().item()
        assert err <= 3 * err32 + 1e-6 * max(1.0, r64.grad.abs().max().item()), (err, err32)
    assert torch.equal(leaves[0].grad, leaves[1].grad)


def test_linear_and_wgrad_random_shapes(pkg):
    """Seeded random problem shapes through whichever kernel the dispatcher picks (A in tensor memory, four
    accumulators for long reductions, split-K): exact on small integers."""
    rng = np.random.default_rng(2024)
    for _ in range(24):
        rows = int(rng.integers(1, 3000))
        in_f = 32 * int(rng.integers(1, 40))
        out_f = 4 * int(rng.integers(1, 100))
        relu = bool(rng.integers(0, 2))
        x = torch.from_numpy(rng.integers(-3, 4, (rows, in_f)).astype(np.float32)).to(DEV)
        w = torch.from_numpy(rng.integers(-3, 4, (out_f, in_f)).astype(np.float32)).to(DEV)
        b = torch.from_numpy(rng.integers(-5, 6, (out_f,)).astype(np.float32)).to(DEV) if rng.integers(0, 2) else None
        ref = x.double() @ w.double().t() + (b.double() if b is not None else 0)
        ref = ref.relu() if relu else ref
        y = pkg.linear_tf32x3(x, w, b, relu=relu)
        assert torch.equal(y, ref.float()), (rows, out_f, in_f, relu)
        gy = torch.from_numpy(rng.integers(-2, 3, (rows, out_f)).astype(np.float32)).to(DEV)
        xs = x[:, : 4 * int(rng.integers(1, in_f // 4 + 1))].contiguous()
        gw, gb = pkg.ops.linear_wgrad(gy, xs)
        assert torch.equal(gw, (gy.double().t() @ xs.double()).float()), (rows, out_f, xs.shape)
        assert torch.equal(gb, gy.double().sum(0).float())


# ---------------------------------------------------------------- fused GroupNorm (SURVEY 8f.4)
@pytest.mark.parametrize("shape,groups,relu,up", [
    ((2, 64, 12, 20), 32, False, None),          # input projection of the small decoder
    ((2, 256, 16, 24), 32, True, None),          # output convolution: GroupNorm + ReLU
    ((3, 256, 24, 40), 32, False, (12, 20)),     # lateral: GroupNorm + up-sampled add (x2)
    ((1, 64, 10, 28), 8, True, (7, 9)),          # odd up-sampling ratio, 8 channels per group
    ((2, 256, 96, 160), 32, False, (48, 80)),    # larger map: several parts per plane
    ((2, 64, 12, 39), 32, False, None),          # KITTI pyramid: W not a multiple of 4 (H*W is)
    ((1, 256, 24, 78), 32, True, None),
])
def test_group_norm_kernel_matches_torch(pkg, shape, groups, relu, up):
    """ops.group_norm == F.group_norm [+ ReLU] [+ F.interpolate(bilinear, align_corners=False)] against
    an fp64 evaluation, no worse than torch's own fp32 kernels (x 2 + 1e-6)."""
    gen = torch.Generator().manual_seed(hash((shape, groups)) % 1000)
    x = (torch.randn(shape, generator=gen) * 2.0 + 3.0).to(DEV)           # mean >> 0: the cancellation case
    norm = torch.nn.GroupNorm(groups, shape[1]).to(DEV)
    with torch.no_grad():
        norm.weight.normal_(1.0, 0.3, generator=None)
        norm.bias.normal_(0.0, 0.5)
    u = torch.randn(shape[0], shape[1], *up, generator=gen).to(DEV) if up else None

    def ref(dtype):
        n = torch.nn.GroupNorm(groups, shape[1]).to(DEV, dtype)
        n.load_state_dict({k: v.to(dtype) for k, v in norm.state_dict().items()})
        r = n(x.to(dtype))
        if relu:
            r = torch.relu(r)
        if u is not None:
            r = r + torch.nn.functional.interpolate(u.to(dtype), size=shape[-2:], mode="bilinear", align_corners=False)
        return r
    with torch.no_grad():
        n0 = pkg.launch_count()
        got = pkg.group_norm(x, norm, relu=relu, up=u)
        assert pkg.launch_count() - n0 == 2
        want64, want32 = ref(torch.float64), ref(torch.float32)
    err = (got.double() - want64).abs().max().item()
    err32 = (want32.double() - want64).abs().max().item()
    assert err <= 2 * err32 + 1e-6, (err, err32)
    with torch.no_grad():                       # deterministic (no atomics)
        assert torch.equal(got, pkg.group_norm(x, norm, relu=relu, up=u))


def test_group_norm_unsupported_shapes_fall_back_in_the_mirror(pkg):
    norm = torch.nn.GroupNorm(4, 8).to(DEV)
    x = torch.randn(1, 8, 5, 7, device=DEV)                 # H*W not a multiple of 4
    assert not pkg.ops.group_norm_supported(x, norm)
    wide = torch.randn(1, 8, 4, 6, device=DEV)              # W % 4 != 0: fine alone, not with the up-sampled add
    assert pkg.ops.group_norm_supported(wide, norm)
    assert not pkg.ops.group_norm_supported(wide, norm, torch.randn(1, 8, 2, 3, device=DEV))
    with pytest.raises(RuntimeError, match="group_norm needs"):
        pkg.group_norm(x, norm)
    conv = pkg.pixel_decoder._ConvNormAct(8, 8, kernel_size=1, norm=norm, activation=torch.nn.functional.relu).to(DEV)
    with torch.no_grad():
        a = conv(x, fused_norm=True)
        b = torch.relu(norm(torch.nn.functional.conv2d(x, conv.weight, conv.bias)))
    assert torch.allclose(a, b, atol=1e-6)


@pytest.mark.parametrize("bias", ["float64", "cpu"])
def test_group_norm_is_not_supported_without_an_fp32_bias_on_the_map_device(pkg, bias):
    """The kernels read the GroupNorm's bias through a raw fp32 pointer on x's device: any other bias is refused
    (the decoder then takes torch's path)."""
    norm = torch.nn.GroupNorm(32, 64).to(DEV)
    b = norm.bias.detach()
    norm.bias = torch.nn.Parameter(b.double() if bias == "float64" else b.cpu())
    x = torch.randn(2, 64, 8, 12, device=DEV)
    assert not pkg.ops.group_norm_supported(x, norm)
    assert not pkg.ops.group_norm_rows_supported(x, norm, torch.empty(2, 8 * 12, 64, device=DEV))
    with pytest.raises(RuntimeError, match="group_norm needs"):
        pkg.group_norm(x, norm)


@pytest.mark.parametrize("shape,groups", [((2, 64, 12, 20), 32), ((3, 256, 8, 16), 32), ((1, 32, 4, 4), 8)])
def test_group_norm_with_the_convolution_bias_folded_in(pkg, shape, groups):
    """ops.group_norm(x, norm, channel_bias=b) == norm(x + b[None, :, None, None]) (fp64 reference)."""
    torch.manual_seed(sum(shape))
    x = torch.randn(*shape, device=DEV) * 2.0 + 0.5
    cb = torch.randn(shape[1], device=DEV) * 3.0
    norm = torch.nn.GroupNorm(groups, shape[1]).to(DEV)
    with torch.no_grad():
        norm.weight.normal_()
        norm.bias.normal_()
        want = F.group_norm((x + cb.view(1, -1, 1, 1)).double(), groups, norm.weight.double(), norm.bias.double(), norm.eps)
        n0 = pkg.launch_count()
        got = pkg.group_norm(x, norm, channel_bias=cb)
        assert pkg.launch_count() - n0 == 2
        assert (got.double() - want).abs().max().item() <= 1e-5
        relu = pkg.group_norm(x, norm, relu=True, channel_bias=cb)
        assert (relu.double() - want.clamp_min(0)).abs().max().item() <= 1e-5
    with pytest.raises(RuntimeError, match="channel_bias must be"):
        pkg.group_norm(x, norm, channel_bias=cb[:-1])


def test_add_channel_bias_in_place(pkg):
    x = torch.randn(3, 40, 6, 10, device=DEV)
    b = torch.randn(40, device=DEV)
    want = x + b.view(1, -1, 1, 1)
    n0 = pkg.launch_count()
    got = pkg.ops.add_channel_bias_(x, b)
    assert pkg.launch_count() - n0 == 1 and got.data_ptr() == x.data_ptr()
    assert torch.equal(got, want)
    assert not pkg.ops.channel_bias_supported(torch.randn(1, 4, 3, 3, device=DEV), torch.randn(4, device=DEV))
    with pytest.raises(RuntimeError, match="add_channel_bias_ needs"):
        pkg.ops.add_channel_bias_(torch.randn(1, 4, 3, 3, device=DEV), torch.randn(4, device=DEV))
    big = torch.randn(2, 8, 256, 512, device=DEV)
    bb = torch.randn(8, device=DEV)
    assert torch.equal(pkg.ops.add_channel_bias_(big.clone(), bb), big + bb.view(1, -1, 1, 1))


def test_transpose_into_destination(pkg):
    x = torch.randn(333, 64, device=DEV)
    dst = torch.empty(64, 333, device=DEV)
    got = pkg.ops.transpose2d(x, out=dst)
    assert got.data_ptr() == dst.data_ptr() and torch.equal(dst, x.t())


@pytest.mark.parametrize("shape,groups,bias", [((2, 64, 12, 20), 32, True), ((3, 256, 8, 16), 32, False),
                                               ((1, 32, 6, 10), 8, True), ((2, 256, 24, 78), 32, True),
                                               ((1, 64, 40, 52), 16, False)])
def test_group_norm_written_as_rows_of_the_concatenated_tensor(pkg, shape, groups, bias):
    """ops.group_norm_rows writes norm(x + b)[n, c, p] to rows[n, p, c] of a slice of a larger [N, S, C] tensor
    (the layout `src.flatten(2).transpose(1, 2)` + `cat` produces) and touches nothing else."""
    torch.manual_seed(sum(shape))
    N, C, H, W = shape
    x = torch.randn(*shape, device=DEV) * 1.5 + 0.25
    cb = torch.randn(C, device=DEV) if bias else None
    norm = torch.nn.GroupNorm(groups, C).to(DEV)
    with torch.no_grad():
        norm.weight.normal_()
        norm.bias.normal_()
        ref_in = x if cb is None else x + cb.view(1, -1, 1, 1)
        want = F.group_norm(ref_in.double(), groups, norm.weight.double(), norm.bias.double(), norm.eps)
        want = want.flatten(2).transpose(1, 2)                         # [N, H*W, C]
        S, start = H * W + 96, 64
        flat = torch.full((N, S, C), -7.0, device=DEV)
        rows = flat[:, start:start + H * W]
        assert pkg.ops.group_norm_rows_supported(x, norm, rows)
        n0 = pkg.launch_count()
        got = pkg.ops.group_norm_rows(x, norm, rows, channel_bias=cb)
        assert pkg.launch_count() - n0 == 2 and got.data_ptr() == rows.data_ptr()
        assert (rows.double() - want).abs().max().item() <= 1e-5
        assert bool((flat[:, :start] == -7.0).all()) and bool((flat[:, start + H * W:] == -7.0).all())
        # the same values as the NCHW kernel, bit for bit
        assert torch.equal(rows, pkg.group_norm(x, norm, channel_bias=cb).flatten(2).transpose(1, 2))
        relu = pkg.ops.group_norm_rows(x, norm, torch.empty(N, H * W, C, device=DEV), channel_bias=cb, relu=True)
        assert (relu.double() - want.clamp_min(0)).abs().max().item() <= 1e-5
    # a wider row stride is fine (rows of a larger tensor); a channel stride other than 1 is not
    wide = torch.empty(N, H * W, C + 4, device=DEV)[..., :C]
    with torch.no_grad():
        assert torch.equal(pkg.ops.group_norm_rows(x, norm, wide, channel_bias=cb), rows)
    assert not pkg.ops.group_norm_rows_supported(x, norm, torch.empty(N, C, H * W, device=DEV).transpose(1, 2))
    with pytest.raises(RuntimeError, match="group_norm_rows needs"):
        pkg.ops.group_norm_rows(x, norm, torch.empty(N, H * W + 1, C, device=DEV))


def test_group_norm_rows_needs_32_channel_blocks(pkg):
    norm = torch.nn.GroupNorm(4, 16).to(DEV)
    x = torch.randn(1, 16, 4, 4, device=DEV)
    assert not pkg.ops.group_norm_rows_supported(x, norm, torch.empty(1, 16, 16, device=DEV))


def test_presplit_weight_gives_the_same_bits_with_one_launch(pkg):
    x, w, b = case(900, 256, 256, seed=21)
    want = pkg.linear_tf32x3(x, w, b, relu=True)
    n0 = pkg.launch_count()
    split = pkg.ops.split_weight(w)
    assert pkg.launch_count() - n0 == 1 and split.numel() == 2 * w.numel()
    n0 = pkg.launch_count()
    got = pkg.linear_tf32x3(x, w, b, relu=True, presplit=split)
    assert pkg.launch_count() - n0 == 1
    assert torch.equal(got, want)
    xl, wl, bl = case(130, 256, 1024, seed=22)                         # long reduction (chunked accumulation)
    assert torch.equal(pkg.linear_tf32x3(xl, wl, bl, presplit=pkg.ops.split_weight(wl)), pkg.linear_tf32x3(xl, wl, bl))
    with pytest.raises(RuntimeError, match="presplit must be"):
        pkg.linear_tf32x3(x, w, b, presplit=split[:-4])
    # the mirror caches the split per weight version
    lin = torch.nn.Linear(256, 256).to(DEV)
    with torch.no_grad():
        n0 = pkg.launch_count()
        y1 = pkg.modules._linear(lin, x, "tf32x3")
        n1 = pkg.launch_count()
        y2 = pkg.modules._linear(lin, x, "tf32x3")
        n2 = pkg.launch_count()
        lin.weight.mul_(2.0)                                            # in-place update: the split is rebuilt
        y3 = pkg.modules._linear(lin, x, "tf32x3")
        n3 = pkg.launch_count()
    assert (n1 - n0, n2 - n1, n3 - n2) == (2, 1, 2) and torch.equal(y1, y2)
    assert (y3 - (2.0 * (y1 - lin.bias) + lin.bias)).abs().max().item() <= 1e-4
