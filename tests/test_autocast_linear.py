"""linear="autocast" on the CPU: every mirror accepts it, and on CPU tensors (no CUDA autocast, so it means
linear="tf32x3", whose kernels take CUDA tensors only) it computes exactly what linear="torch" does; unknown values and
amp=True with linear="tf32x3" still raise."""
import pytest
import torch

LEVELS = [(2, 3), (4, 6), (8, 12)]


def oracle_core(oracle):
    def core(value, shapes, lsi, loc, w, im2col_step):
        return oracle.core_grid_sample(value, shapes, loc, w)
    return core


def test_encoder_mirrors_accept_autocast_and_match_torch_on_cpu(pkg, oracle):
    kw = dict(d_model=64, nhead=2, num_encoder_layers=2, dim_feedforward=128, dropout=0.0,
              num_feature_levels=3, enc_n_points=4, core=oracle_core(oracle))
    torch.manual_seed(5)
    a = pkg.modules.MSDeformAttnTransformerEncoderOnly(**kw).eval()
    b = pkg.modules.MSDeformAttnTransformerEncoderOnly(linear="autocast", **kw).eval()
    b.load_state_dict(a.state_dict())
    assert all(layer.linear == "autocast" and layer.self_attn.linear == "autocast" for layer in b.encoder.layers)
    srcs = [torch.randn(2, 64, h, w) for h, w in LEVELS]
    pos = [torch.randn(2, 64, h, w) for h, w in LEVELS]
    with torch.no_grad():
        assert torch.equal(a(srcs, pos)[0], b(srcs, pos)[0])
    ya, yb = a(srcs, pos)[0], b(srcs, pos)[0]                      # autograd on
    assert torch.equal(ya, yb)
    ya.square().sum().backward()
    yb.square().sum().backward()
    for (n, p), (_, q) in zip(a.named_parameters(), b.named_parameters()):
        assert torch.equal(p.grad, q.grad), n


def test_pixel_decoder_accepts_autocast_and_matches_torch_on_cpu(pkg, oracle):
    from test_pixel_decoder import build
    a, feats, _ = build(pkg, core=oracle_core(oracle))
    b, _, _ = build(pkg, core=oracle_core(oracle), linear="autocast")
    with torch.no_grad():
        ra, rb = a.forward_features(feats), b.forward_features(feats)
    for x, y in zip([ra[0], ra[1], *ra[2]], [rb[0], rb[1], *rb[2]]):
        assert torch.equal(x, y)


def test_amp_pixel_decoder_accepts_autocast_and_still_refuses_tf32x3(pkg):
    from test_pixel_decoder import PD_KW, PD_SHAPES
    m = pkg.pixel_decoder.MSDeformAttnPixelDecoder(PD_SHAPES, linear="autocast", amp=True, **PD_KW)
    assert m.amp and m.linear == "autocast"
    with pytest.raises(ValueError, match="tf32x3"):
        pkg.pixel_decoder.MSDeformAttnPixelDecoder(PD_SHAPES, linear="tf32x3", amp=True, **PD_KW)


def test_unknown_linear_value_still_raises(pkg):
    with pytest.raises(ValueError, match="unknown linear implementation"):
        pkg.modules._linear(torch.nn.Linear(4, 4), torch.randn(2, 4), "fp8")
    layer = torch.nn.Linear(4, 4)
    x = torch.randn(2, 4)
    assert torch.equal(pkg.modules._linear(layer, x, "autocast"), layer(x))


def test_mixed_wrappers_refuse_cpu_tensors(pkg):
    x, w = torch.randn(8, 128), torch.randn(128)
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        pkg.add_layernorm_mixed(x, x.bfloat16(), w, w)
    assert not pkg.ops.add_layernorm_mixed_supported(x, x.bfloat16(), w, w)
    assert not pkg.ops.add_layernorm_mixed_backward_supported(x, x.bfloat16(), w)
    assert not pkg.ops.ms_deform_attn_fused_mixed_forward_packed_supported(
        torch.randn(1, 4, 1, 32).bfloat16(), torch.rand(1, 4, 1, 2), torch.randn(1, 4, 12).bfloat16(), 1, 4)
