"""Mirror of the reference's MSDeformAttnPixelDecoder (uni-encoder-code_b200/pixel_decoder.py) against
the committed golden of the reference class (tests/golden/make_golden.py::pixel_decoder_golden):
parameter names, init, forward_features."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from test_modules import assert_state_equals_golden, oracle_core, redraw_attention_projections

PD_KW = dict(transformer_dropout=0.0, transformer_nheads=2, transformer_dim_feedforward=96,
             transformer_enc_layers=2, conv_dim=64, mask_dim=32, norm="GN",
             transformer_in_features=["res3", "res4", "res5"], common_stride=4)
PD_SHAPES = {"res2": (12, 4), "res3": (20, 8), "res4": (28, 16), "res5": (36, 32)}


def build(pkg, core=None, device="cpu", fused=False, linear="torch"):
    g = load_golden("pixel_decoder_small")
    m = pkg.pixel_decoder.MSDeformAttnPixelDecoder(PD_SHAPES, core=core, fused=fused, linear=linear, **PD_KW)
    state = {k[len("state::"):]: torch.from_numpy(v) for k, v in g.items() if k.startswith("state::")}
    missing, unexpected = m.load_state_dict(state, strict=True)
    assert not missing and not unexpected
    feats = {k[len("feat::"):]: torch.from_numpy(v).to(device) for k, v in g.items() if k.startswith("feat::")}
    return m.to(device).eval(), feats, g


def check(outs, g, tol):
    mask_feat, low, multi = outs
    assert tuple(mask_feat.shape) == g["mask_features"].shape and len(multi) == 3
    assert np.abs(mask_feat.detach().cpu().numpy() - g["mask_features"]).max() <= tol
    assert np.abs(low.detach().cpu().numpy() - g["lowest"]).max() <= tol
    for i, m in enumerate(multi):
        assert np.abs(m.detach().cpu().numpy() - g[f"multi{i}"]).max() <= tol


def test_mirror_loads_reference_checkpoint_and_matches_forward_features_cpu(pkg, oracle):
    m, feats, g = build(pkg, core=oracle_core(oracle))
    with torch.no_grad():
        check(m.forward_features(feats), g, 2e-5)
    # the position embedding is input-independent and cached per shape
    assert len(m.pe_layer._cache) == 3


def test_mirror_init_matches_reference_pixel_decoder_golden(pkg):
    """The golden's weights are the reference decoder's init under torch.manual_seed(4321), its attention
    projections then redrawn, and its features come from the same generator (make_golden.py
    pixel_decoder_golden): under the same seed the mirror reproduces the parameter order and every
    tensor bit for bit.  (The sine embedding is pinned by test_modules.py.)"""
    g = load_golden("pixel_decoder_small")
    torch.manual_seed(4321)
    m = pkg.pixel_decoder.MSDeformAttnPixelDecoder(PD_SHAPES, **PD_KW)
    gen = torch.Generator().manual_seed(77)
    redraw_attention_projections(m.transformer.encoder.layers, gen, torch.float32)
    assert_state_equals_golden(m, g)
    for k, (c, s) in PD_SHAPES.items():
        assert np.array_equal(torch.randn(2, c, 64 // s, 96 // s, generator=gen).numpy(), g["feat::" + k])


@pytest.mark.gpu
@pytest.mark.parametrize("fused,linear", [(False, "torch"), (True, "torch"), (False, "tf32x3"), (True, "tf32x3")])
def test_mirror_plus_cuda_op_matches_reference_pixel_decoder_golden(pkg, fused, linear):
    m, feats, g = build(pkg, device="cuda:0", fused=fused, linear=linear)
    n0 = pkg.launch_count()
    # cuDNN convolutions default to TF32 on this GPU (1e-3 errors); the golden is true fp32
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            outs = m.forward_features(feats)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    # one MSDA forward per encoder layer (+ weight split and GEMM for each of the 6 linears of a layer;
    # conv_dim 64 is not a width the fused residual + LayerNorm kernel covers, so torch runs those;
    # + statistics and apply kernel of the fused GroupNorm for the four maps whose plane is a multiple
    # of 4 here: the stride-8 and stride-16 input projections, the lateral and the output convolution at stride 4;
    # + one transpose per image for the NCHW copy of the finest encoder level + the mask_features bias)
    # with fused=True (2 heads of 32 channels: the fused kernels apply) the two query projections are ONE stacked
    # GEMM on `src` (its weight split once, + the table GEMM on the first call): 5 + 6 instead of 6 x 2 per layer
    n_img = next(iter(feats.values())).shape[0]
    per_layer = 1 + (5 + 6 if fused else 6 * 2)
    assert pkg.launch_count() - n0 == (2 if linear == "torch" else 2 * per_layer + 4 * 2 + n_img + 1)
    check(outs, g, 5e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("fused,linear", [(False, "torch"), (True, "tf32x3")])
def test_forward_features_is_cuda_graph_capturable(pkg, fused, linear):
    """No host read of device data and no host-to-device copy is left in the mirror's forward (position
    embeddings, reference points and the level tensors are cached per shape), so the whole call records
    into one CUDA graph; the replay reproduces the eager result bit for bit."""
    m, feats, g = build(pkg, device="cuda:0", fused=fused, linear=linear)
    with torch.no_grad():
        eager = m.forward_features(feats)            # also fills the per-shape caches
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            m.forward_features(feats)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = m.forward_features(feats)
        for k in feats:
            feats[k].add_(0.0)                       # inputs stay where they are; replay reads them again
        graph.replay()
        torch.cuda.synchronize()
    assert torch.equal(out[0], eager[0]) and torch.equal(out[1], eager[1])
    for a, b in zip(out[2], eager[2]):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_inference_kernels_under_inference_mode_and_repeated_calls(pkg):
    """The inference path (fused kernels, cached tables) gives the same bits under torch.inference_mode() as under
    no_grad, call after call (the caches are keyed on tensor versions, which inference tensors do not have)."""
    m, feats, g = build(pkg, device="cuda:0", fused=True, linear="tf32x3")
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False          # the golden is true fp32 (cuDNN convolutions default to TF32)
    try:
        with torch.no_grad():
            a = m.forward_features(feats)
        with torch.inference_mode():
            b = m.forward_features(feats)
            c = m.forward_features({k: v.clone() for k, v in feats.items()})
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    for x, y, z in zip([a[0], a[1], *a[2]], [b[0], b[1], *b[2]], [c[0], c[1], *c[2]]):
        assert torch.equal(x, y) and torch.equal(x, z)
    check(b, g, 5e-4)


@pytest.mark.gpu
def test_full_width_decoder_with_every_inference_kernel_matches_the_torch_path(pkg):
    """conv_dim 256 / 8 heads (32 channels per head, the shape the fused kernels cover): GroupNorm written as
    rows of the concatenated tensor, `src + pos` folded into the per-query table, stacked query GEMM read in
    place, channel bias, transposes -- all on, against the same weights on torch's fp32 kernels."""
    torch.manual_seed(5)
    kw = dict(transformer_dropout=0.0, transformer_nheads=8, transformer_dim_feedforward=1024,
              transformer_enc_layers=2, conv_dim=256, mask_dim=256, norm="GN",
              transformer_in_features=["res3", "res4", "res5"], common_stride=4)
    shapes = {"res2": (96, 4), "res3": (192, 8), "res4": (384, 16), "res5": (768, 32)}
    ref = pkg.pixel_decoder.MSDeformAttnPixelDecoder(shapes, **kw).cuda().eval()
    fast = pkg.pixel_decoder.MSDeformAttnPixelDecoder(shapes, fused=True, linear="tf32x3", **kw).cuda().eval()
    for m in ref.modules():                                    # away from the zero-initialised producers
        if isinstance(m, pkg.modules.MSDeformAttn):
            torch.nn.init.normal_(m.sampling_offsets.weight, std=0.02)
            torch.nn.init.normal_(m.attention_weights.weight, std=0.05)
    fast.load_state_dict(ref.state_dict())
    feats = {k: torch.randn(2, c, 128 // s, 256 // s, device="cuda:0") for k, (c, s) in shapes.items()}
    tf32_conv, tf32_mm = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            want = ref.forward_features(feats)
            n0 = pkg.launch_count()
            got = fast.forward_features(feats)
            first = pkg.launch_count() - n0
            n0 = pkg.launch_count()
            again = fast.forward_features(feats)
            steady = pkg.launch_count() - n0
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32_conv, tf32_mm
    # per layer: fused forward + 5 GEMMs + 2 x add-LayerNorm; 5 GroupNorms x 2; 2 transposes; bias; the first call
    # also splits the weights (4 Linears + the stacked query weight per layer) and builds the query tables (a GEMM each)
    assert steady == 2 * (1 + 5 + 2) + 5 * 2 + 2 + 1 and first == steady + 2 * (5 + 1)
    for a, b, c in zip([want[0], want[1], *want[2]], [got[0], got[1], *got[2]], [again[0], again[1], *again[2]]):
        assert torch.equal(b, c)
        assert (a - b).abs().max().item() <= 2e-4 * max(1.0, a.abs().max().item()), (a - b).abs().max().item()


@pytest.mark.gpu
def test_caches_are_not_filled_during_graph_capture(pkg):
    """A graph captured on a model whose per-module caches (split weights, query tables, position rows, sine
    embedding) are still cold must not leave un-materialised tensors in them: an eager call after the capture, and
    the replay, both give the result of a normally warmed model."""
    warm, feats, g = build(pkg, device="cuda:0", fused=True, linear="tf32x3")
    cold, _, _ = build(pkg, device="cuda:0", fused=True, linear="tf32x3")
    with torch.no_grad():
        want = warm.forward_features(feats)            # also fills the module-global shape caches (host -> device copies)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            torch.zeros(1, device="cuda:0")            # the side stream exists and is idle
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = cold.forward_features(feats)
        eager = cold.forward_features(feats)           # right after the capture, before any replay
        graph.replay()
        torch.cuda.synchronize()
    for a, b, c in zip([want[0], want[1], *want[2]], [eager[0], eager[1], *eager[2]], [out[0], out[1], *out[2]]):
        assert torch.equal(a, b) and torch.equal(a, c)
