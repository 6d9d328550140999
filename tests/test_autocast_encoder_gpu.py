"""The encoder under torch.autocast on the library's kernels (linear="autocast").

Kernel contracts, bit for bit:
* add_layernorm_mixed: y == add_layernorm(x, residual.float()) and y16 == y.to(dtype);
* add_layernorm_mixed_backward: with g = grad_y + grad_y16.float(), grad_x == add_layernorm_backward(g, x,
  residual.float()) and grad_residual == grad_x.to(dtype); the deterministic twin equals the fp32 twin on g;
* ms_deform_attn_fused_mixed_forward_packed == round16(fp32 packed forward on the widened inputs, same table).
Modules: without an active 16-bit autocast linear="autocast" is linear="tf32x3" bit for bit; under one, the pixel
decoder is held to the bar of test_mixed_precision_gpu (what the composition moves when every input moves by one
16-bit ulp) against linear="torch" with the up-cast oracle core.
"""
import contextlib
import os
import subprocess
import sys

import pytest
import torch

from test_fused_gpu import make_case
from test_fused_mixed_gpu import assert_bits
from test_mixed_precision_gpu import _nrel, _upcast_oracle_core, deterministic_mode, ulp16

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DTYPES = [torch.bfloat16, torch.float16]
ERR_NULL, ERR_SHAPE, ERR_UNSUPPORTED = -1, -2, -3
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def ln_case(rows, cols, dtype, seed=0, scale=1.0):
    gen = torch.Generator().manual_seed(seed)
    x = (torch.randn(rows, cols, generator=gen) * 2 + 0.5).to(DEV)
    res = (torch.randn(rows, cols, generator=gen) * scale).to(dtype).to(DEV)
    w = (torch.rand(cols, generator=gen) + 0.5).to(DEV)
    b = (torch.randn(cols, generator=gen) * 0.1).to(DEV)
    return x, res, w, b


def same16(a, b):
    """16-bit tensors equal element for element (inf included; NaN where the other is NaN)."""
    assert a.dtype == b.dtype
    assert torch.equal(a.isnan(), b.isnan())
    assert torch.equal(torch.nan_to_num(a.float(), nan=0.0, posinf=1e30, neginf=-1e30),
                       torch.nan_to_num(b.float(), nan=0.0, posinf=1e30, neginf=-1e30))


# ---------------------------------------------------------------- 1. residual + LayerNorm, forward
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("cols", [128, 256, 384, 512])
@pytest.mark.parametrize("rows", [1, 1003, 65536 + 5])
def test_add_layernorm_mixed_forward(pkg, dtype, cols, rows):
    x, res, w, b = ln_case(rows, cols, dtype, seed=cols + rows)
    if rows > 8:                                     # non-finite inputs: the affected rows only
        x[3, 7] = float("inf")
        x[5, 1] = float("nan")
        res[6, 2] = float("-inf")
    y, y16 = pkg.add_layernorm_mixed(x, res, w, b, 1e-5)
    want = pkg.add_layernorm(x, res.float(), w, b, 1e-5)
    assert_bits(y, want, "y")
    same16(y16, y.to(dtype))
    y_only, none = pkg.add_layernorm_mixed(x, res, w, b, 1e-5, want_y16=False)
    assert none is None and torch.equal(y_only.nan_to_num(), y.nan_to_num())


def test_fp16_y16_overflow_is_inf(pkg):
    x, res, w, b = ln_case(1003, 256, torch.float16, seed=3)
    w = w * 1e5                                      # |y| well above 65504
    y, y16 = pkg.add_layernorm_mixed(x, res, w, b, 1e-5)
    assert torch.isfinite(y).all() and torch.isinf(y16).any()
    same16(y16, y.to(torch.float16))


@pytest.mark.parametrize("dtype", DTYPES)
def test_misaligned_views(pkg, dtype):
    """A 16-bit residual view that is not 8-byte aligned: MSDA_ERR_UNSUPPORTED at the ABI, torch's composition in the
    module."""
    rows, cols = 257, 256
    x, res, w, b = ln_case(rows, cols, dtype, seed=9)
    buf = torch.empty(rows * cols + 1, dtype=dtype, device=DEV)
    view = buf[1:].view(rows, cols)
    view.copy_(res)
    y = torch.empty_like(x)
    fn = {torch.bfloat16: pkg._lib.lib.msda_b200_add_layernorm_mixed_bf16,
          torch.float16: pkg._lib.lib.msda_b200_add_layernorm_mixed_f16}[dtype]
    stream = torch.cuda.current_stream().cuda_stream
    assert fn(x.data_ptr(), view.data_ptr(), w.data_ptr(), b.data_ptr(), y.data_ptr(), None, rows, cols, 1e-5,
              stream) == ERR_UNSUPPORTED
    assert fn(x.data_ptr(), None, w.data_ptr(), b.data_ptr(), y.data_ptr(), None, rows, cols, 1e-5,
              stream) == ERR_NULL
    assert fn(x.data_ptr(), res.data_ptr(), w.data_ptr(), b.data_ptr(), y.data_ptr(), None, rows, 192, 1e-5,
              stream) == ERR_UNSUPPORTED
    assert fn(x.data_ptr(), res.data_ptr(), w.data_ptr(), b.data_ptr(), y.data_ptr(), None, 0, cols, 1e-5,
              stream) == ERR_SHAPE
    assert not pkg.ops.add_layernorm_mixed_supported(x, view, w, b, need_bias=True)
    norm = torch.nn.LayerNorm(cols).to(DEV)
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        got, copy = pkg.modules._add_norm_mixed(norm, x, view)
        want = norm(x + view)
    assert copy is None and torch.equal(got, want)


# ---------------------------------------------------------------- 2. backward
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("cols", [128, 256])
@pytest.mark.parametrize("which", ["both", "y", "y16"])
def test_add_layernorm_mixed_backward(pkg, dtype, cols, which):
    rows = 20003
    x, res, w, _ = ln_case(rows, cols, dtype, seed=cols)
    gen = torch.Generator().manual_seed(7)
    gy = torch.randn(rows, cols, generator=gen).to(DEV) if which != "y16" else None
    gy16 = torch.randn(rows, cols, generator=gen).to(dtype).to(DEV) if which != "y" else None
    gx, gr, gg, gb = pkg.ops.add_layernorm_mixed_backward(gy, gy16, x, res, w, 1e-5)
    g = gy + gy16.float() if which == "both" else (gy if gy is not None else gy16.float())
    want_x, want_g, want_b = pkg.ops.add_layernorm_backward(g.contiguous(), x, res.float(), w, 1e-5)
    assert torch.equal(gx, want_x)
    same16(gr, gx.to(dtype))
    for got, want in ((gg, want_g), (gb, want_b)):          # reduction order of the atomics
        assert torch.allclose(got, want, rtol=1e-5, atol=1e-5 * want.abs().max().item())


@pytest.mark.parametrize("dtype", DTYPES)
def test_add_layernorm_mixed_backward_deterministic(pkg, dtype):
    rows, cols = 40000 + 3, 256
    x, res, w, _ = ln_case(rows, cols, dtype, seed=1)
    gen = torch.Generator().manual_seed(2)
    gy = torch.randn(rows, cols, generator=gen).to(DEV)
    gy16 = torch.randn(rows, cols, generator=gen).to(dtype).to(DEV)
    with deterministic_mode():
        a = pkg.ops.add_layernorm_mixed_backward(gy, gy16, x, res, w, 1e-5)
        b = pkg.ops.add_layernorm_mixed_backward(gy, gy16, x, res, w, 1e-5)
        want = pkg.ops.add_layernorm_backward(gy + gy16.float(), x, res.float(), w, 1e-5)
    for p, q in zip(a, b):
        assert torch.equal(p, q)
    assert torch.equal(a[0], want[0]) and torch.equal(a[2], want[1]) and torch.equal(a[3], want[2])
    same16(a[1], a[0].to(dtype))


@pytest.mark.parametrize("dtype", DTYPES)
def test_function_matches_autocast_composition_gradients(pkg, dtype):
    """AddLayerNormMixedFunction: the forward and gradients of torch's composition `layer_norm(x + r)` and its cast,
    with either output unused."""
    rows, cols = 1003, 256
    x0, r0, w0, b0 = ln_case(rows, cols, dtype, seed=4)
    for use in ("both", "y", "y16"):
        leaves = [t.clone().requires_grad_(True) for t in (x0, r0, w0, b0)]
        ref_leaves = [t.clone().requires_grad_(True) for t in (x0, r0, w0, b0)]
        y, y16 = pkg.AddLayerNormMixedFunction.apply(*leaves, 1e-5)
        ry = torch.nn.functional.layer_norm(ref_leaves[0] + ref_leaves[1].float(), (cols,), ref_leaves[2],
                                            ref_leaves[3], 1e-5)
        ry16 = ry.to(dtype)
        assert torch.allclose(y, ry, atol=1e-5, rtol=1e-5)
        loss = (y.square().sum() if use != "y16" else 0) + (y16.float().sum() * 0.5 if use != "y" else 0)
        rloss = (ry.square().sum() if use != "y16" else 0) + (ry16.float().sum() * 0.5 if use != "y" else 0)
        loss.backward()
        rloss.backward()
        assert leaves[1].grad.dtype == dtype and leaves[0].grad.dtype == torch.float32
        for got, want in zip(leaves, ref_leaves):
            assert _nrel(got.grad.float(), want.grad.float()) < 1e-3, use


# ---------------------------------------------------------------- 3. the 16-bit packed / table forward
def _packed_check(pkg, c, dtype, lq=None, table_scale=0.3):
    d = {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in c.items()}
    levels = d["levels"]
    L = len(levels)
    P = d["off"].shape[4]
    M = d["off"].shape[2]
    if lq is not None:
        d["off"], d["logits"], d["ref"] = (d["off"][:, :lq].contiguous(), d["logits"][:, :lq].contiguous(),
                                           d["ref"][:, :lq].contiguous())
    N, Lq = d["off"].shape[:2]
    proj16 = torch.cat((d["off"].reshape(N, Lq, -1), d["logits"].reshape(N, Lq, -1)), -1).to(dtype).contiguous()
    value16 = d["value"].to(dtype)
    table = (torch.randn(Lq, proj16.shape[-1], generator=torch.Generator().manual_seed(Lq)) * table_scale).to(DEV)
    for tab in (None, table):
        want = pkg.ops.ms_deform_attn_fused_forward_packed(value16.float(), d["shapes"], d["lsi"], d["ref"],
                                                           proj16.float(), L, P, query_table=tab).to(dtype)
        n0 = pkg.launch_count()
        got = pkg.ops.ms_deform_attn_fused_mixed_forward_packed(value16, d["shapes"], d["lsi"], d["ref"], proj16, L, P,
                                                                query_table=tab)
        assert pkg.launch_count() - n0 == 1
        assert_bits(got, want, f"table={tab is not None}")
    return d, value16, proj16, table, M, L, P


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("levels,points,shared_ref,lq", [
    ([(12, 20), (6, 10)], 4, True, None),                    # L*P = 8
    ([(16, 16), (8, 8), (4, 4), (2, 2)], 4, False, None),    # L*P = 16, per-image reference points
    ([(9, 13)], 4, True, None),                              # L*P = 4, odd sizes
    ([(16, 32), (8, 16), (4, 8)], 4, True, 301),             # L*P = 12, Lq != S
    ([(16, 32), (8, 16), (4, 8)], 4, False, None),           # L*P = 12, per-image reference points
])
def test_packed_table_forward_bit_identical(pkg, dtype, levels, points, shared_ref, lq):
    c = make_case(pkg, levels, 2, 8, points, shared_ref, seed=5 + len(levels))
    _packed_check(pkg, c, dtype, lq)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name", ["kitti_384x1248_b16", "cityscapes_512x1024_b8", "cityscapes_1024x2048_b8"])
def test_packed_table_forward_full_size(pkg, dtype, name):
    w = pkg.synthetic.WORKLOADS[name]
    c = make_case(pkg, list(w.levels), w.batch, 8, 4, True, seed=3)
    _packed_check(pkg, c, dtype)


@pytest.mark.parametrize("dtype", DTYPES)
def test_packed_table_abi_errors(pkg, dtype):
    """The fp32 strided entry's error codes: bad strides are shape errors, a one-sided table a null pointer."""
    c = make_case(pkg, [(16, 32), (8, 16), (4, 8)], 2, 8, 4, True, seed=11)
    d, value16, proj16, table, M, L, P = _packed_check(pkg, c, dtype)
    N, Lq, width = proj16.shape
    out = torch.empty(N, Lq, M * 32, dtype=dtype, device=DEV)
    fn = {torch.bfloat16: pkg._lib.lib.msda_b200_fused_forward_strided_bf16,
          torch.float16: pkg._lib.lib.msda_b200_fused_forward_strided_f16}[dtype]
    args = lambda so, sl, ot=None, lt=None, off_ptr=proj16.data_ptr(): (
        value16.data_ptr(), d["shapes"].data_ptr(), d["lsi"].data_ptr(), d["ref"].data_ptr(), 0, off_ptr, so,
        proj16.data_ptr() + 2 * M * L * P * 2, sl, ot, lt, N, value16.shape[1], M, 32, L, Lq, P, out.data_ptr(),
        None)
    assert fn(*args(width, width)) == 0
    assert fn(*args(width + 1, width)) == ERR_SHAPE
    assert fn(*args(2 * M * L * P - 2, width)) == ERR_SHAPE
    assert fn(*args(width, M * L * P - 1)) == ERR_SHAPE
    assert fn(*args(width, width, ot=table.data_ptr())) == ERR_NULL
    assert fn(*args(width, width, off_ptr=proj16.data_ptr() + 2)) == ERR_UNSUPPORTED     # offsets pair not 4-aligned
    torch.cuda.synchronize()


# ---------------------------------------------------------------- 4. encoder and pixel decoder
SHAPES = {"res2": (32, 4), "res3": (48, 8), "res4": (64, 16), "res5": (96, 32)}
KW = dict(transformer_dropout=0.0, transformer_nheads=4, transformer_dim_feedforward=256, transformer_enc_layers=2,
          conv_dim=128, mask_dim=64, norm="GN", transformer_in_features=["res3", "res4", "res5"], common_stride=4)


def _decoder(pkg, linear, fused=True, amp=True, core=None):
    torch.manual_seed(0)
    m = pkg.pixel_decoder.MSDeformAttnPixelDecoder(SHAPES, core=core, fused=fused, linear=linear, amp=amp, **KW)
    # the reference init zeroes the offset / attention weights: every sampling point would sit exactly on a bilinear
    # cell edge (offsets from the bias only), where the location gradient changes with the side a kernel picks
    gen = torch.Generator().manual_seed(3)
    with torch.no_grad():
        for layer in m.transformer.encoder.layers:
            for lin in (layer.self_attn.sampling_offsets, layer.self_attn.attention_weights):
                lin.weight.copy_(torch.randn(lin.weight.shape, generator=gen) * 0.02)
    return m.to(DEV).eval()


def _features(seed=1, n=2, h=128, w=256):
    gen = torch.Generator().manual_seed(seed)
    return {k: torch.randn(n, c, h // s, w // s, generator=gen).to(DEV) for k, (c, s) in SHAPES.items()}


def _flat(o):
    return [o[0], o[1], *o[2]]


def _step(m, feats, dtype, weights, scaler_ctx=None):
    m.zero_grad(set_to_none=True)
    ctx = torch.autocast("cuda", dtype=dtype) if dtype is not None else contextlib.nullcontext()
    with ctx:
        outs = _flat(m.forward_features(feats))
    loss = sum((o.float() * w).sum() for o, w in zip(outs, weights))
    loss.backward()
    grads = {n: p.grad.float().clone() for n, p in m.named_parameters() if p.grad is not None}
    return [o.detach().float() for o in outs], grads


def _weights(m, feats, seed=21):
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        shapes = [o.shape for o in _flat(m.forward_features(feats))]
    return [torch.randn(s, generator=gen).to(DEV) for s in shapes]


def _fresh_process(call):
    """`call` (source of a call of a function of this module) in a new Python process whose environment has
    CUBLAS_WORKSPACE_CONFIG set from its start -> its last line of output.  torch's cuBLAS GEMMs are reproducible in
    deterministic mode only with it, and setting it here would change the cuBLAS kernels of every other test."""
    code = (f"import sys; sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]\n"
            f"import test_autocast_encoder_gpu as t\nprint(t.{call})")
    env = dict(os.environ)
    env.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    args = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    res = subprocess.run(args, env=env, capture_output=True, text=True, timeout=1200)
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-4000:]
    return res.stdout.strip().splitlines()[-1]


def tf32x3_equivalence(amp):
    """The inference forward, and a training step in deterministic mode (the tf32x3 weight-gradient and LayerNorm
    backward kernels reduce with atomics otherwise), of linear="autocast" with no autocast active against
    linear="tf32x3" -> "same" when every output and gradient is bit-identical."""
    from __graft_entry__ import load_package
    pkg = load_package()
    feats = _features()
    a = _decoder(pkg, "autocast", amp=amp)
    b = _decoder(pkg, "tf32x3", amp=False)
    with torch.no_grad():
        for x, y in zip(_flat(a.forward_features(feats)), _flat(b.forward_features(feats))):
            assert torch.equal(x, y)
    weights = _weights(b, feats)
    torch.backends.cudnn.deterministic = True
    with deterministic_mode():
        oa, ga = _step(a.train(), feats, None, weights)
        ob, gb = _step(b.train(), feats, None, weights)
    assert set(ga) == set(gb)
    assert all(torch.equal(x, y) for x, y in zip(oa, ob))
    assert all(torch.equal(ga[n], gb[n]) for n in ga), [n for n in ga if not torch.equal(ga[n], gb[n])]
    return "same"


@pytest.mark.parametrize("amp", [False, True])
def test_without_autocast_bit_identical_to_tf32x3(amp):
    assert _fresh_process(f"tf32x3_equivalence({amp})") == "same"


def _perturbed(feats, dtype, seed=5):
    gen = torch.Generator().manual_seed(seed)
    out = {}
    for k, v in feats.items():
        sign = torch.where(torch.rand(v.shape, generator=gen) < 0.5, -1.0, 1.0).to(DEV)
        out[k] = v + sign * torch.from_numpy(ulp16(v.cpu().numpy(), dtype)).float().to(DEV)
    return out


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("fused", [True, False])
def test_pixel_decoder_under_autocast(pkg, oracle, dtype, fused):
    feats = _features()
    m = _decoder(pkg, "autocast", fused=fused).train()
    ref = _decoder(pkg, "torch", fused=False, core=_upcast_oracle_core(oracle)).train()
    weights = _weights(ref, feats)
    timing = pkg.ops.enable_timing(True)
    try:
        outs, grads = _step(m, feats, dtype, weights)
        kinds = {k for k, _, _ in timing}
    finally:
        pkg.ops.enable_timing(False)
    assert {"add_layernorm_mixed", "add_layernorm_mixed_backward"} <= kinds, kinds
    ref_outs, ref_grads = _step(ref, feats, dtype, weights)
    p_outs, p_grads = _step(ref, _perturbed(feats, dtype), dtype, weights)
    assert set(grads) == set(ref_grads)
    for i, (o, r, p) in enumerate(zip(outs, ref_outs, p_outs)):
        assert torch.isfinite(o).all()
        assert _nrel(o, r) <= _nrel(p, r), f"output {i}: {_nrel(o, r)} > {_nrel(p, r)}"
    for n in grads:
        assert torch.isfinite(grads[n]).all(), n
        assert _nrel(grads[n], ref_grads[n]) <= _nrel(p_grads[n], ref_grads[n]), \
            f"{n}: {_nrel(grads[n], ref_grads[n])} > {_nrel(p_grads[n], ref_grads[n])}"
    # inference: the forward alone, against the same bar
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        got = [o.float() for o in _flat(m.eval().forward_features(feats))]
        want = [o.float() for o in _flat(ref.eval().forward_features(feats))]
        moved = [o.float() for o in _flat(ref.forward_features(_perturbed(feats, dtype)))]
    for i, (o, r, p) in enumerate(zip(got, want, moved)):
        assert _nrel(o, r) <= _nrel(p, r), f"inference output {i}"


@pytest.mark.parametrize("dtype", DTYPES)
def test_folded_position_embedding_under_autocast(pkg, monkeypatch, dtype):
    """Inference with the batch-shared position embedding: one 16-bit query GEMM on src16 and the 16-bit packed
    forward with the fp32 table, held to the bar against the unfolded path of the same module."""
    feats = _features()
    m = _decoder(pkg, "autocast")
    calls = []
    real = pkg.ops.ms_deform_attn_fused_mixed_forward_packed
    monkeypatch.setattr(pkg.ops, "ms_deform_attn_fused_mixed_forward_packed",
                        lambda *a, **k: calls.append(1) or real(*a, **k))
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        folded = [o.float() for o in _flat(m.forward_features(feats))]
    assert len(calls) == KW["transformer_enc_layers"]
    for layer in m.transformer.encoder.layers:
        monkeypatch.setattr(layer.self_attn, "can_fold_pos", lambda *a, **k: False)
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        unfolded = [o.float() for o in _flat(m.forward_features(feats))]
        moved = [o.float() for o in _flat(m.forward_features(_perturbed(feats, dtype)))]
    assert len(calls) == KW["transformer_enc_layers"]
    for i, (o, r, p) in enumerate(zip(folded, unfolded, moved)):
        assert torch.isfinite(o).all()
        assert _nrel(o, r) <= _nrel(p, r), f"output {i}: {_nrel(o, r)} > {_nrel(p, r)}"


@pytest.mark.parametrize("dtype", DTYPES)
def test_autocast_forward_in_a_cuda_graph_replays_bit_identically(pkg, dtype):
    feats = _features()
    m = _decoder(pkg, "autocast")
    static = {k: v.clone() for k, v in feats.items()}
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype, cache_enabled=False):
        eager = [o.clone() for o in _flat(m.forward_features(static))]
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                m.forward_features(static)
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            captured = _flat(m.forward_features(static))
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        for a, b in zip(captured, eager):
            assert torch.equal(a, b)


def encoder_steps_twice(dtype_name):
    """Two training steps of the autocast encoder (linear="autocast", fused producers) under
    torch.use_deterministic_algorithms(True) and cudnn.deterministic -> "same" when outputs and gradients match."""
    from __graft_entry__ import load_package
    pkg = load_package()
    dtype = getattr(torch, dtype_name)
    torch.manual_seed(0)
    m = pkg.modules.MSDeformAttnTransformerEncoderOnly(d_model=256, nhead=8, num_encoder_layers=2,
                                                       dim_feedforward=512, dropout=0.0, num_feature_levels=3,
                                                       enc_n_points=4, fused=True, linear="autocast").to(DEV).train()
    levels = [(16, 32), (8, 16), (4, 8)]
    gen = torch.Generator().manual_seed(1)
    srcs = [torch.randn(2, 256, h, w, generator=gen).to(DEV) for h, w in levels]
    pos = [torch.randn(2, 256, h, w, generator=gen).to(DEV) for h, w in levels]
    proj = torch.randn(2, sum(h * w for h, w in levels), 256, generator=gen).to(DEV)

    def step():
        m.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=dtype):
            out = m(srcs, pos)[0]
        (out.float() * proj).sum().backward()
        return out.detach().clone(), {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}

    torch.backends.cudnn.deterministic = True
    timing = pkg.ops.enable_timing(True)
    with deterministic_mode():
        (o1, g1), (o2, g2) = step(), step()
    kinds = {k for k, _, _ in timing}
    pkg.ops.enable_timing(False)
    assert "add_layernorm_mixed_backward" in kinds, kinds
    assert torch.equal(o1, o2)
    assert set(g1) == set(g2) and all(torch.equal(g1[n], g2[n]) for n in g1), [n for n in g1 if not torch.equal(g1[n], g2[n])]
    return "same"


@pytest.mark.parametrize("dtype", DTYPES)
def test_deterministic_training_steps(dtype):
    assert _fresh_process(f"encoder_steps_twice({str(dtype).split('.')[-1]!r})") == "same"
