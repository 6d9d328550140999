"""Host-side mirrors of the callers (uni-encoder-code_b200/modules.py) against the reference's own
classes: parameter names / init / forward on CPU (core op injected from the oracle: test
infrastructure), and mirror + CUDA op on the GPU against the committed encoder golden."""
import numpy as np
import pytest
import torch

from conftest import load_golden
import ref_import

LEVELS = [(2, 3), (4, 6), (8, 12)]


def oracle_core(oracle):
    def core(value, shapes, lsi, loc, w, im2col_step):
        return oracle.core_grid_sample(value, shapes, loc, w)
    return core


def build_small(pkg, core=None, dtype=torch.float64, device="cpu"):
    m = pkg.modules.MSDeformAttnTransformerEncoderOnly(
        d_model=64, nhead=2, num_encoder_layers=2, dim_feedforward=128, dropout=0.0,
        num_feature_levels=3, enc_n_points=4, core=core)
    g = load_golden("encoder_small")
    state = {k[len("state::"):]: torch.from_numpy(v) for k, v in g.items() if k.startswith("state::")}
    m = m.double()                      # load at full precision, then cast
    missing, unexpected = m.load_state_dict(state, strict=True)
    assert not missing and not unexpected
    return m.to(device=device, dtype=dtype).eval(), g


def test_mirror_loads_reference_checkpoint_and_matches_reference_forward_cpu(pkg, oracle):
    m, g = build_small(pkg, core=oracle_core(oracle))
    srcs = [torch.from_numpy(g[f"src{i}"]) for i in range(3)]
    srcs[2].requires_grad_(True)
    pos = [torch.from_numpy(g[f"pos{i}"]) for i in range(3)]
    memory, shapes, lsi, vr = m(srcs, pos)
    assert shapes.tolist() == g["spatial_shapes"].tolist() and lsi.tolist() == g["level_start_index"].tolist()
    assert torch.equal(vr, torch.ones_like(vr))
    assert (memory.detach().numpy() - g["memory"]).__abs__().max() <= 1e-11
    (memory * torch.from_numpy(g["cotangent"])).sum().backward()
    assert np.abs(srcs[2].grad.numpy() - g["grad_src2"]).max() <= 1e-10


def redraw_attention_projections(layers, gen, dtype):
    """What tests/golden/make_golden.py does to the reference's seeded init before it stores the weights:
    sampling offsets and attention weights of every layer redrawn from `gen`, so that the locations leave
    the integer pixel steps of the default init."""
    with torch.no_grad():
        for layer in layers:
            a = layer.self_attn
            a.sampling_offsets.weight.copy_(torch.randn(a.sampling_offsets.weight.shape, generator=gen, dtype=dtype) * 0.05)
            a.sampling_offsets.bias.add_(torch.rand(a.sampling_offsets.bias.shape, generator=gen, dtype=dtype) * 0.6 + 0.2)
            a.attention_weights.weight.copy_(torch.randn(a.attention_weights.weight.shape, generator=gen, dtype=dtype) * 0.1)


def assert_state_equals_golden(module, g):
    state = module.state_dict()
    assert list(state) == [k[len("state::"):] for k in g if k.startswith("state::")]
    for k, v in state.items():
        assert np.array_equal(v.numpy(), g["state::" + k]), k


def test_mirror_init_matches_reference_golden(pkg):
    """The golden's weights are the reference encoder's init under torch.manual_seed(1234), redrawn as
    above, and its inputs come from the same generator (make_golden.py encoder_golden): under the same
    seed the mirror reproduces the parameter order and every tensor bit for bit, and its sine position
    embedding reproduces the reference's `pos` inputs."""
    g = load_golden("encoder_small")
    torch.manual_seed(1234)
    m = pkg.modules.MSDeformAttnTransformerEncoderOnly(
        d_model=64, nhead=2, num_encoder_layers=2, dim_feedforward=128, dropout=0.0,
        num_feature_levels=3, enc_n_points=4).double()
    gen = torch.Generator().manual_seed(99)
    redraw_attention_projections(m.encoder.layers, gen, torch.float64)
    assert_state_equals_golden(m, g)
    pe = pkg.pixel_decoder.PositionEmbeddingSine(32, normalize=True)
    for i, (h, w) in enumerate(LEVELS):
        src = torch.randn(2, 64, h, w, generator=gen, dtype=torch.float64)
        assert np.array_equal(src.numpy(), g[f"src{i}"])
        assert np.array_equal(pe(src).double().numpy(), g[f"pos{i}"])


def test_reference_points_match_reference_formula(pkg):
    enc = pkg.modules.MSDeformAttnTransformerEncoder
    shapes = torch.tensor(LEVELS)
    vr = torch.rand(2, 3, 2) * 0.5 + 0.5
    got = enc.get_reference_points(shapes, vr, "cpu")
    # restated from msdeformattn.py:152-166
    want = []
    for lvl, (H, W) in enumerate(LEVELS):
        ys, xs = torch.meshgrid(torch.linspace(0.5, H - 0.5, H), torch.linspace(0.5, W - 0.5, W), indexing="ij")
        y = ys.reshape(-1)[None] / (vr[:, None, lvl, 1] * H)
        x = xs.reshape(-1)[None] / (vr[:, None, lvl, 0] * W)
        want.append(torch.stack((x, y), -1))
    want = torch.cat(want, 1)[:, :, None] * vr[:, None]
    assert torch.allclose(got, want, atol=1e-6)
    ones = pkg.modules.reference_points_for(LEVELS, "cpu").expand(2, -1, -1, -1)
    assert torch.allclose(enc.get_reference_points(shapes, torch.ones(2, 3, 2), "cpu"), ones, atol=1e-7)


@pytest.mark.skipif(not ref_import.available(), reason="reference checkout not present")
def test_mirror_init_and_forward_equal_live_reference(pkg, oracle):
    """Same seed -> same parameters as the reference classes; same forward on CPU."""
    ns = ref_import.load()
    kw = dict(d_model=64, nhead=2, num_encoder_layers=2, dim_feedforward=128, dropout=0.0,
              num_feature_levels=3, enc_n_points=4)
    torch.manual_seed(7)
    ref = ns.MSDeformAttnTransformerEncoderOnly(**kw).eval()
    torch.manual_seed(7)
    mine = pkg.modules.MSDeformAttnTransformerEncoderOnly(core=oracle_core(oracle), **kw).eval()
    rs, ms = ref.state_dict(), mine.state_dict()
    assert list(rs) == list(ms)
    for k in rs:
        assert torch.equal(rs[k], ms[k]), k
    srcs = [torch.randn(2, 64, h, w) for h, w in LEVELS]
    pe = ns.PositionEmbeddingSine(32, normalize=True)
    pos = [pe(s) for s in srcs]
    with torch.no_grad():
        a = ref(srcs, pos)[0]
        b = mine(srcs, pos)[0]
    assert (a - b).abs().max().item() <= 2e-5

    # module level: the reference MSDeformAttn CPU branch (ms_deform_attn.py:122-124) vs the mirror
    torch.manual_seed(3)
    r_attn = ns.MSDeformAttn(64, 3, 2, 4).double()
    m_attn = pkg.modules.MSDeformAttn(64, 3, 2, 4, core=oracle_core(oracle)).double()
    m_attn.load_state_dict(r_attn.state_dict())
    q = torch.randn(2, 126, 64, dtype=torch.float64)
    x = torch.randn(2, 126, 64, dtype=torch.float64)
    refp = torch.rand(2, 126, 3, 2, dtype=torch.float64)
    shapes = torch.tensor(LEVELS)
    lsi = torch.tensor([0, 6, 30])
    mask = torch.rand(2, 126) > 0.8
    with torch.no_grad():
        assert (r_attn(q, refp, x, shapes, lsi, mask) - m_attn(q, refp, x, shapes, lsi, mask)).abs().max() <= 1e-12
        box = torch.rand(2, 126, 3, 4, dtype=torch.float64)      # 4-d reference boxes (ms_deform_attn.py:113-115)
        assert (r_attn(q, box, x, shapes, lsi) - m_attn(q, box, x, shapes, lsi)).abs().max() <= 1e-12


def test_module_padding_mask_and_box_reference_points(pkg, oracle):
    """The two module inputs the encoder never passes: a padding mask zeroes the value rows it marks, so
    those rows of `input_flatten` cannot reach the output; 4-d reference boxes (cx, cy, w, h) give
    loc = (cx, cy) + offset / P * (w, h) / 2 (ms_deform_attn.py:113-115)."""
    seen = {}

    def core(value, shapes, lsi, loc, w, im2col_step):
        seen["loc"] = loc
        return oracle.core_grid_sample(value, shapes, loc, w)
    torch.manual_seed(3)
    attn = pkg.modules.MSDeformAttn(64, 3, 2, 4, core=core).double()
    with torch.no_grad():
        attn.sampling_offsets.weight.normal_(std=0.05)
        q = torch.randn(2, 126, 64, dtype=torch.float64)
        x = torch.randn(2, 126, 64, dtype=torch.float64)
        shapes, lsi = torch.tensor(LEVELS), torch.tensor([0, 6, 30])
        refp = torch.rand(2, 126, 3, 2, dtype=torch.float64)
        mask = torch.rand(2, 126) > 0.8
        y = attn(q, refp, x, shapes, lsi, mask)
        assert torch.equal(attn(q, refp, x + 5.0 * mask[..., None], shapes, lsi, mask), y)
        assert not torch.equal(attn(q, refp, x + 5.0 * ~mask[..., None], shapes, lsi, mask), y)
        box = torch.rand(2, 126, 3, 4, dtype=torch.float64)
        attn(q, box, x, shapes, lsi)
        off = attn.sampling_offsets(q).view(2, 126, 2, 3, 4, 2)
        want = box[:, :, None, :, None, :2] + off / 4 * box[:, :, None, :, None, 2:] * 0.5
        assert (seen["loc"] - want).abs().max().item() <= 1e-15


def test_module_refuses_cpu_without_injected_core(pkg):
    m = pkg.modules.MSDeformAttn(64, 3, 2, 4)
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        m(torch.randn(1, 126, 64), torch.rand(1, 126, 3, 2), torch.randn(1, 126, 64),
          torch.tensor(LEVELS), torch.tensor([0, 6, 30]))


def test_inference_kernel_option_is_inert_on_cpu_and_wrappers_refuse_cpu(pkg, oracle):
    """linear="tf32x3" selects CUDA kernels for CUDA tensors only: on CPU tensors (host-logic tests with an
    injected core) the mirror takes torch's kernels and gives the very same numbers; the wrappers themselves
    refuse CPU tensors like the reference's extension does."""
    kw = dict(d_model=64, nhead=2, num_encoder_layers=2, dim_feedforward=128, dropout=0.0,
              num_feature_levels=3, enc_n_points=4, core=oracle_core(oracle))
    torch.manual_seed(3)
    a = pkg.modules.MSDeformAttnTransformerEncoderOnly(**kw).eval()
    b = pkg.modules.MSDeformAttnTransformerEncoderOnly(linear="tf32x3", **kw).eval()
    b.load_state_dict(a.state_dict())
    srcs = [torch.randn(1, 64, h, w) for h, w in LEVELS]
    pos = [torch.randn(1, 64, h, w) for h, w in LEVELS]
    with torch.no_grad():
        assert torch.equal(a(srcs, pos)[0], b(srcs, pos)[0])
    assert torch.equal(a(srcs, pos)[0], b(srcs, pos)[0])            # autograd on
    with pytest.raises(ValueError, match="unknown linear implementation"):
        pkg.modules._linear(torch.nn.Linear(4, 4), torch.randn(2, 4), "fp8")
    x, w = torch.randn(8, 32), torch.randn(8, 32)
    for call in (lambda: pkg.linear_tf32x3(x, w, None), lambda: pkg.add_layernorm(x, None, w[0], w[1]),
                 lambda: pkg.ops.linear_wgrad(x, x)):
        with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
            call()
    # the level tensors are cached per (pyramid, device) and equal the reference's construction
    shapes, lsi = pkg.modules.level_tensors_for(LEVELS, "cpu")
    assert shapes.tolist() == [list(l) for l in LEVELS] and lsi.tolist() == [0, 6, 30]
    assert pkg.modules.level_tensors_for(LEVELS, "cpu")[0] is shapes


@pytest.mark.gpu
def test_mirror_plus_cuda_op_matches_reference_encoder_golden(pkg):
    """Reference encoder (fp64, CPU, in the build container) vs mirror + sm_100a kernels in fp32."""
    m, g = build_small(pkg, dtype=torch.float32, device="cuda:0")
    srcs = [torch.from_numpy(g[f"src{i}"]).float().cuda() for i in range(3)]
    srcs[2].requires_grad_(True)
    pos = [torch.from_numpy(g[f"pos{i}"]).float().cuda() for i in range(3)]
    memory = m(srcs, pos)[0]
    assert np.abs(memory.detach().double().cpu().numpy() - g["memory"]).max() <= 2e-4
    (memory * torch.from_numpy(g["cotangent"]).float().cuda()).sum().backward()
    ref = g["grad_src2"]
    assert np.abs(srcs[2].grad.double().cpu().numpy() - ref).max() <= 2e-4 * max(1.0, np.abs(ref).max())


@pytest.mark.gpu
def test_mirror_fp64_cuda_op_matches_reference_encoder_golden(pkg):
    m, g = build_small(pkg, dtype=torch.float64, device="cuda:0")
    srcs = [torch.from_numpy(g[f"src{i}"]).cuda() for i in range(3)]
    pos = [torch.from_numpy(g[f"pos{i}"]).cuda() for i in range(3)]
    with torch.no_grad():
        memory = m(srcs, pos)[0]
    assert np.abs(memory.cpu().numpy() - g["memory"]).max() <= 1e-9


def test_inference_position_cache_tracks_its_inputs(pkg, oracle):
    """In inference the (position + level) embedding is cached; new position tensors, an in-place change of
    them or of level_embed must all invalidate it."""
    m = pkg.modules.MSDeformAttnTransformerEncoderOnly(d_model=64, nhead=2, num_encoder_layers=1, dim_feedforward=64,
                                                       dropout=0.0, num_feature_levels=3, enc_n_points=4,
                                                       core=oracle_core(oracle)).eval()
    srcs = [torch.randn(1, 64, h, w) for h, w in LEVELS]

    def fresh(pos):
        m._pos_cache_key = None
        with torch.no_grad():
            return m(srcs, pos)[0]
    with torch.no_grad():
        for _ in range(3):
            pos = [torch.randn(1, 64, h, w) for h, w in LEVELS]
            assert torch.equal(m(srcs, pos)[0], fresh(pos))
            assert torch.equal(m(srcs, pos)[0], fresh(pos))          # second call: served from the cache
            pos[1].mul_(2.0)
            assert torch.equal(m(srcs, pos)[0], fresh(pos))
            m.level_embed.add_(0.5)
            assert torch.equal(m(srcs, pos)[0], fresh(pos))
    assert torch.equal(m(srcs, pos)[0], fresh(pos))                   # autograd on: no cache involved


def test_encoder_and_pixel_decoder_run_under_inference_mode(pkg, oracle):
    """The reference works under torch.inference_mode(); inference tensors do not track ._version, so
    the mirror's position cache must not read it (advisor finding, round 1)."""
    m, g = build_small(pkg, core=oracle_core(oracle))
    srcs = [torch.from_numpy(g[f"src{i}"]) for i in range(3)]
    pos = [torch.from_numpy(g[f"pos{i}"]) for i in range(3)]
    with torch.no_grad():
        want = m(srcs, pos)[0]
    with torch.inference_mode():
        got = m([s.clone() for s in srcs], [p.clone() for p in pos])[0]     # inference tensors as inputs
        again = m(srcs, pos)[0]
    assert torch.equal(got, want) and torch.equal(again, want)
    from test_pixel_decoder import build
    dec, feats, _ = build(pkg, core=oracle_core(oracle))
    with torch.no_grad():
        ref_out = dec.forward_features(feats)
    with torch.inference_mode():
        out = dec.forward_features({k: v.clone() for k, v in feats.items()})
    assert torch.equal(out[0], ref_out[0]) and torch.equal(out[1], ref_out[1])


def test_shape_keyed_caches_are_bounded(pkg):
    """Variable-resolution datasets present thousands of pyramids: the device-side constants cached per
    shape (reference points, level tensors, sine embeddings) must not grow without bound."""
    mod = pkg.modules
    for i in range(40):
        levels = [(2 + i, 3), (4, 5 + i)]
        mod.reference_points_for(levels, "cpu")
        mod.level_tensors_for(levels, "cpu")
    assert len(mod._REF_CACHE) <= mod._REF_CACHE.maxsize <= 16
    assert len(mod._LEVEL_CACHE) <= mod._LEVEL_CACHE.maxsize <= 16
    pe = pkg.pixel_decoder.PositionEmbeddingSine(8, normalize=True)
    for i in range(40):
        pe(torch.zeros(1, 1, 3 + i, 4))
    assert len(pe._cache) <= pe._cache.maxsize <= 16
    a = pe(torch.zeros(1, 1, 5, 4))
    assert torch.equal(a, pe(torch.zeros(2, 1, 5, 4))[:1])                 # hit == rebuilt


def test_batch_shared_position_embedding_and_preflattened_input_on_cpu(pkg, oracle):
    """Host logic of the round-2 inference path, without a GPU: a position embedding shared by the batch
    (stride 0) stays ONE copy of the rows broadcast over the batch; the folded-projection path and the split-weight
    cache never engage on the CPU; pre-flattened rows give the same result as the per-level maps."""
    m, g = build_small(pkg, core=oracle_core(oracle), dtype=torch.float32)
    srcs = [torch.from_numpy(g[f"src{i}"]).float() for i in range(3)]
    one = [torch.from_numpy(g[f"pos{i}"]).float()[:1] for i in range(3)]
    n = srcs[0].shape[0]
    shared = [p.expand(n, -1, -1, -1) for p in one]
    copies = [p.expand(n, -1, -1, -1).contiguous() for p in one]
    with torch.no_grad():
        src, pos, shapes, lsi, levels = m.flatten_inputs(srcs, shared)
        assert pos.shape[0] == n and pos.stride(0) == 0 and pos[0].is_contiguous()
        src2, pos2, _, _, _ = m.flatten_inputs(srcs, copies)
        assert pos2.stride(0) != 0 and torch.equal(pos.contiguous(), pos2)
        layer = m.encoder.layers[0]
        ref = pkg.modules.reference_points_for(levels, "cpu").expand(n, -1, -1, -1)
        assert not layer.self_attn.can_fold_pos(src, pos, ref)          # CPU tensors, linear="torch"
        a = m(srcs, shared)[0]
        b = m(srcs, copies)[0]
        c = m(None, shared, src_flat=src.clone(), levels=levels)[0]
    assert torch.equal(a, b) and torch.equal(a, c)
    # with autograd on, the embedding is materialised per image as the reference does
    src3, pos3, _, _, _ = m.flatten_inputs(srcs, shared)
    assert pos3.stride(0) != 0
    assert "_tf32x3_presplit" not in layer.linear1.__dict__
