"""The mixed-precision fused-producer MSDA op: bf16 / fp16 value, raw sampling offsets, attention logits and their
gradients, fp32 reference points, every quantity in between in fp32.

Contract: for the same widened inputs the fp32 arithmetic is the fp32 fused kernels' instruction sequence, and each
output is rounded once.  So output, grad_sampling_offsets, grad_attn_logits (every backward kernel) and the
deterministic grad_value are bit-identical to round16(fp32 fused op on the widened inputs); the default grad_value
depends on reduction order, as in fp32, and is held to one 16-bit ulp of it.
"""
import numpy as np
import pytest
import torch

from conftest import FWD_ABS_TOL, GRAD_REL_TOL
from test_fused_gpu import make_case, reference_composition
from test_mixed_precision_gpu import deterministic_mode, option, ulp16, widened

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DTYPES = [torch.bfloat16, torch.float16]
SHAPES = [   # those of test_fused_gpu.test_fused_matches_unfused_composition
    ([(8, 16), (16, 32), (32, 64)], 2, 8, 4, True),      # pixel-decoder shape, L*P = 12
    ([(12, 39), (24, 78)], 1, 4, 4, False),              # odd sizes, per-image reference points, L*P = 8
    ([(7, 9), (5, 3), (4, 4), (2, 2)], 2, 2, 4, True),   # L*P = 16
    ([(9, 13)], 3, 2, 4, True),                          # L*P = 4
]


def rounded(c, dtype):
    """The widened inputs: value and grad_output through test_mixed_precision_gpu.widened, and the fused op's 16-bit
    offsets and logits rounded the same way (all kept as fp32 CPU tensors)."""
    out = widened({**c, "grad_output": c["grad_out"]}, dtype)
    out["grad_out"] = out.pop("grad_output")
    for k in ("off", "logits"):
        out[k] = c[k].to(dtype).float()
    return out


def to_dev(c, dtype=None):
    """On the device; with `dtype`, value / off / logits / grad_out in that type (reference points stay fp32)."""
    return {k: (v.to(dtype) if dtype is not None and k in ("value", "off", "logits", "grad_out") else v).to(DEV)
            .contiguous() if torch.is_tensor(v) else v for k, v in c.items()}


def run_fused(pkg, d):
    """Forward + backward of MSDeformAttnFusedFunction -> (output, grad_value, grad_offsets, grad_logits)."""
    # detach(), not clone(): the leaves keep the inputs' storage, so a deliberately offset view stays offset
    value = d["value"].detach().requires_grad_(True)
    off = d["off"].detach().requires_grad_(True)
    logits = d["logits"].detach().requires_grad_(True)
    out = pkg.MSDeformAttnFusedFunction.apply(value, d["shapes"], d["lsi"], d["ref"], off, logits)
    out.backward(d["grad_out"])
    torch.cuda.synchronize()
    return out.detach(), value.grad, off.grad, logits.grad


def excess(got, ref, dtype, tol):
    """max(|got - ref| - (ulp16(ref) + tol * max|ref|)); <= 0 passes.  NaN / inf must sit in the same places."""
    g = got.double().cpu().numpy() if torch.is_tensor(got) else np.asarray(got, dtype=np.float64)
    r = np.asarray(ref.double().cpu().numpy() if torch.is_tensor(ref) else ref, dtype=np.float64).reshape(g.shape)
    fin = np.isfinite(r)
    assert np.array_equal(np.isfinite(g), fin) and np.array_equal(g[~fin], r[~fin], equal_nan=True)
    if not fin.any():
        return 0.0
    d = np.abs(g[fin] - r[fin]) - (ulp16(r[fin], dtype) + tol * np.abs(r[fin]).max())
    return float(d.max())


def assert_bits(a, b, what):
    assert a.dtype == b.dtype, what
    assert torch.equal(a.isnan(), b.isnan()), what
    assert torch.equal(torch.nan_to_num(a), torch.nan_to_num(b)), what


def check_against_fp32_fused(pkg, c, dtype, det=False):
    """The 16-bit fused op on `c` rounded to `dtype` against round16(fp32 fused op on the widened inputs)."""
    w = rounded(c, dtype)
    want = [t.to(dtype) for t in run_fused(pkg, to_dev(w))]
    got = run_fused(pkg, to_dev(c, dtype))
    for g, wt, name in zip(got, want, ("output", "grad_value", "grad_offsets", "grad_logits")):
        assert g.dtype == dtype, name
        if name == "grad_value" and not det:
            # the default grad_value: fp32 reductions in a scheduling-dependent order, then one rounding
            assert excess(g, wt, dtype, 1e-5) <= 0, name
        else:
            assert_bits(g, wt, name)
    return got


# ---------------------------------------------------------------- 1. bit identity with the fp32 fused op
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("levels,batch,heads,points,shared_ref", SHAPES)
@pytest.mark.parametrize("bwd_variant", [0, 20, 2])   # probe-gated default, merging kernel forced, per-row kernel forced
def test_bit_identical_to_rounded_fp32_fused(pkg, levels, batch, heads, points, shared_ref, bwd_variant, dtype):
    c = make_case(pkg, levels, batch, heads, points, shared_ref, seed=21)
    with option(pkg, "bwd_variant", bwd_variant):
        check_against_fp32_fused(pkg, c, dtype)
        # launches: those of the plain 16-bit op on the same shape (forward, backward kernel(s), grad_value rounding)
        d = to_dev(c, dtype)
        L = len(levels)
        N, S, M = c["off"].shape[:3]
        wts = torch.softmax(d["logits"].float(), -1).view(N, S, M, L, points)
        loc = d["ref"][:, :, None, :, None, :] + d["off"].float() / d["shapes"].flip(-1).float()[None, None, None, :, None, :]
        n0 = pkg.launch_count()
        run_fused(pkg, d)
        n1 = pkg.launch_count()
        v = d["value"].clone().requires_grad_(True)
        o = pkg.MSDeformAttnMixedFunction.apply(v, d["shapes"], d["lsi"], loc.contiguous(), wts.contiguous(), 128)
        o.backward(d["grad_out"])
        torch.cuda.synchronize()
        assert n1 - n0 == pkg.launch_count() - n1


# ---------------------------------------------------------------- 2. against the fp64 composition
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("levels,batch,heads,points,shared_ref", SHAPES)
def test_matches_fp64_composition_on_widened_inputs(pkg, oracle, levels, batch, heads, points, shared_ref, dtype):
    c = make_case(pkg, levels, batch, heads, points, shared_ref, seed=21)
    w = rounded(c, dtype)
    out, gv, goff, glog = run_fused(pkg, to_dev(c, dtype))
    ref_out, ref_gv, ref_goff, ref_glog = reference_composition(oracle, w)
    assert excess(out, ref_out, dtype, 0) <= 2 * FWD_ABS_TOL
    for got, ref, name in ((gv, ref_gv, "grad_value"), (goff, ref_goff, "grad_offsets"), (glog, ref_glog, "grad_logits")):
        assert excess(got, ref, dtype, GRAD_REL_TOL) <= 0, name


# ---------------------------------------------------------------- 3. against the module's unfused autocast path
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("levels,batch,heads,points,shared_ref", SHAPES[:2])
def test_matches_unfused_autocast_composition(pkg, levels, batch, heads, points, shared_ref, dtype):
    """torch's fp32 softmax and `ref + off.float() / (W, H)` feeding the mixed-precision op, as MSDeformAttn(fused=False)
    runs under autocast; its offsets / logits gradients are rounded back to 16 bits by the upcasts' backward."""
    c = make_case(pkg, levels, batch, heads, points, shared_ref, seed=21)
    d = to_dev(c, dtype)
    out, gv, goff, glog = run_fused(pkg, d)
    v2 = d["value"].clone().requires_grad_(True)
    o2 = d["off"].clone().requires_grad_(True)
    l2 = d["logits"].clone().requires_grad_(True)
    N, S, M = c["off"].shape[:3]
    w = torch.softmax(l2.float(), -1).view(N, S, M, len(levels), points)
    wh = d["shapes"].flip(-1).float()
    loc = d["ref"][:, :, None, :, None, :] + o2.float() / wh[None, None, None, :, None, :]
    out2 = pkg.MSDeformAttnMixedFunction.apply(v2, d["shapes"], d["lsi"], loc.contiguous(), w.contiguous(), 128)
    out2.backward(d["grad_out"])
    assert o2.grad.dtype == dtype and l2.grad.dtype == dtype
    assert excess(out, out2.detach(), dtype, 0) <= 2e-5
    assert excess(gv, v2.grad, dtype, 1e-5) <= 0
    assert excess(glog, l2.grad, dtype, 1e-4) <= 0
    assert excess(goff, o2.grad, dtype, 1e-4) <= 0


# ---------------------------------------------------------------- 4. edges
def edge_case(pkg, levels, batch, heads, points, lq=None, seed=5):
    """Points on cell edges and map borders, off the map, +-inf / NaN offsets, +-inf and +-100 logits."""
    c = make_case(pkg, levels, batch, heads, points, True, seed=seed)
    if lq is not None:
        c["off"], c["logits"], c["ref"] = c["off"][:, :lq], c["logits"][:, :lq], c["ref"][:, :lq].contiguous()
        c["grad_out"] = c["grad_out"][:, :lq]
    off, logits = c["off"].clone(), c["logits"].clone()
    gen = torch.Generator().manual_seed(seed)
    r = torch.rand(off.shape[:-1], generator=gen)
    off[..., 0] = torch.where(r < 0.15, torch.round(off[..., 0]) + 0.5, off[..., 0])    # on a cell edge (the pixel
    off[..., 1] = torch.where(r < 0.15, torch.round(off[..., 1]) + 0.5, off[..., 1])    # centres are at k + 0.5)
    off[..., 0] = torch.where((r > 0.2) & (r < 0.25), off[..., 0] * 300, off[..., 0])   # off the map
    flat = off.view(-1)
    flat[3], flat[40], flat[77], flat[101] = float("inf"), float("-inf"), float("nan"), 1e4
    lflat = logits.view(-1)
    lflat[5], lflat[17], lflat[29], lflat[30] = 100.0, -100.0, float("inf"), float("-inf")
    lflat[logits.shape[-1] * 7 + 2] = float("-inf")          # one row with a -inf logit only
    c["off"], c["logits"] = off.contiguous(), logits.contiguous()
    c["grad_out"] = c["grad_out"].contiguous()
    return c


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("lq", [None, 301])             # encoder (Lq == S) and decoder-style queries
@pytest.mark.parametrize("bwd_variant", [0, 2])
def test_edges(pkg, dtype, lq, bwd_variant):
    c = edge_case(pkg, [(16, 32), (8, 16), (4, 8)], 2, 8, 4, lq=lq)
    with option(pkg, "bwd_variant", bwd_variant):
        check_against_fp32_fused(pkg, c, dtype)
        with deterministic_mode():
            check_against_fp32_fused(pkg, c, dtype, det=True)


def test_fp16_offset_gradient_overflow_is_inf(pkg):
    """A grad_sampling_offsets beyond the fp16 range comes out +-inf (GradScaler's signal), as round16 of fp32."""
    c = make_case(pkg, [(8, 16), (4, 8)], 1, 2, 4, True, seed=2)
    c["value"] = c["value"] * 6e3
    c["grad_out"] = c["grad_out"] * 6e3
    _, _, goff, glog = check_against_fp32_fused(pkg, c, torch.float16)
    assert torch.isinf(goff).any()


# ---------------------------------------------------------------- 5. full size
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name", ["cityscapes_512x1024_b8", "kitti_384x1248_b16"])
def test_full_size(pkg, name, dtype):
    """BASELINE configs[1] and the KITTI batch-16 shape."""
    w = pkg.synthetic.WORKLOADS[name]
    c = make_case(pkg, list(w.levels), w.batch, 8, 4, True, seed=3)
    check_against_fp32_fused(pkg, c, dtype)


# ---------------------------------------------------------------- 6. alignment
def _offset_view(t, elements):
    buf = torch.empty(t.numel() + elements, dtype=t.dtype, device=t.device)
    return buf[elements:].view(t.shape).copy_(t)


@pytest.mark.parametrize("dtype", DTYPES)
def test_value_view_16_but_not_64_byte_aligned_takes_the_per_row_kernel(pkg, dtype):
    c = make_case(pkg, [(16, 32), (8, 16), (4, 8)], 2, 8, 4, True, seed=7)
    w = rounded(c, dtype)
    with option(pkg, "bwd_variant", 2):                      # the fp32 reference on the same (per-row) kernel
        want = [t.to(dtype) for t in run_fused(pkg, to_dev(w))]
    d = to_dev(c, dtype)
    d["value"] = _offset_view(d["value"], 8)                 # 16 bytes into an allocation
    assert d["value"].data_ptr() % 16 == 0 and d["value"].data_ptr() % 64 != 0
    n0 = pkg.launch_count()
    out, gv, goff, glog = run_fused(pkg, d)
    assert pkg.launch_count() - n0 == 3                      # forward, per-row backward, grad_value rounding
    assert_bits(out, want[0], "output")
    assert_bits(goff, want[2], "grad_offsets")
    assert_bits(glog, want[3], "grad_logits")
    assert excess(gv, want[1], dtype, 1e-5) <= 0


@pytest.mark.parametrize("dtype", DTYPES)
def test_rejected_views_behave_as_the_fp32_fused_op(pkg, dtype):
    """A value view the 32-channel kernels cannot read: the fused entries refuse it in both precisions."""
    c = make_case(pkg, [(8, 16), (4, 8)], 1, 2, 4, True, seed=8)
    for dt in (torch.float32, dtype):
        d = to_dev(c, dt)
        d["value"] = _offset_view(d["value"], 1)
        with pytest.raises(RuntimeError, match="unsupported"):
            pkg.ms_deform_attn_fused_forward(d["value"], d["shapes"], d["lsi"], d["ref"], d["off"], d["logits"])
    # 16-bit offsets one element into their storage: not 4-byte aligned for the pair loads
    d = to_dev(c, dtype)
    d["off"] = _offset_view(d["off"], 1)
    with pytest.raises(RuntimeError, match="unsupported"):
        pkg.ms_deform_attn_fused_forward(d["value"], d["shapes"], d["lsi"], d["ref"], d["off"], d["logits"])


# ---------------------------------------------------------------- 7. determinism and CUDA graphs
def _backward(pkg, d):
    return pkg.ops.ms_deform_attn_fused_backward(d["value"], d["shapes"], d["lsi"], d["ref"], d["off"], d["logits"],
                                                 d["grad_out"])


def _captured(pkg, fn):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        res = fn()
    graph.replay()
    torch.cuda.synchronize()
    return res


@pytest.mark.parametrize("dtype", DTYPES)
def test_deterministic_mode(pkg, monkeypatch, dtype):
    levels = [(16, 32), (8, 16), (4, 8)]
    c = make_case(pkg, levels, 2, 8, 4, False, seed=13)
    d = to_dev(c, dtype)
    w = to_dev(rounded(c, dtype))
    with deterministic_mode():
        n0 = pkg.launch_count()
        g1 = _backward(pkg, d)
        assert pkg.launch_count() - n0 == 4                 # records, sort, bounds, gather: no accumulation buffer
        g2 = _backward(pkg, d)
        gg = _captured(pkg, lambda: _backward(pkg, d))
        S = sum(h * wd for h, wd in levels)
        monkeypatch.setattr(pkg.ops, "DETERMINISTIC_RECORD_LIMIT", S * 8 * len(levels) * 4 * 4)
        g3 = _backward(pkg, d)
        want = [t.to(dtype) for t in _backward(pkg, w)]
    for other in (g2, gg, g3, want):
        for x, y in zip(g1, other):
            assert_bits(x, y, "deterministic")


@pytest.mark.parametrize("dtype", DTYPES)
def test_graph_replay_default_mode(pkg, dtype):
    d = to_dev(make_case(pkg, [(16, 32), (8, 16), (4, 8)], 2, 8, 4, True, seed=17), dtype)
    fwd = lambda: pkg.ms_deform_attn_fused_forward(d["value"], d["shapes"], d["lsi"], d["ref"], d["off"], d["logits"])
    eager_out, eager = fwd(), _backward(pkg, d)
    out = _captured(pkg, fwd)
    gv, goff, glog = _captured(pkg, lambda: _backward(pkg, d))
    assert_bits(out, eager_out, "output")
    assert_bits(goff, eager[1], "grad_offsets")
    assert_bits(glog, eager[2], "grad_logits")
    assert excess(gv, eager[0].float(), dtype, 1e-5) <= 0


# ---------------------------------------------------------------- 8. dtype contract
def test_dtype_contract(pkg):
    c = make_case(pkg, [(8, 16), (4, 8)], 1, 2, 4, True, seed=4)
    for dtype in DTYPES:
        other = torch.float16 if dtype == torch.bfloat16 else torch.bfloat16
        d = to_dev(c, dtype)
        bad = [(dict(d, off=d["off"].to(other)), "sampling_offsets"),
               (dict(d, ref=d["ref"].to(dtype)), "reference_points"),
               (dict(d, off=d["off"].float()), "sampling_offsets"),
               (dict(d, logits=d["logits"].float()), "attn_logits")]
        for b, name in bad:
            with pytest.raises(RuntimeError, match=name):
                pkg.ms_deform_attn_fused_forward(b["value"], b["shapes"], b["lsi"], b["ref"], b["off"], b["logits"])
            assert not pkg.ops.fused_supported(b["value"], b["ref"], b["off"], b["logits"])
        with pytest.raises(RuntimeError, match="grad_output"):
            pkg.ops.ms_deform_attn_fused_backward(d["value"], d["shapes"], d["lsi"], d["ref"], d["off"], d["logits"],
                                                  d["grad_out"].to(other))
        # the packed projection forward stays fp32
        N, Lq = d["off"].shape[:2]
        proj = torch.cat((d["off"].reshape(N, Lq, -1), d["logits"].reshape(N, Lq, -1)), -1).contiguous()
        with pytest.raises(RuntimeError, match="fused MSDA covers"):
            pkg.ops.ms_deform_attn_fused_forward_packed(d["value"], d["shapes"], d["lsi"], d["ref"], proj, 2, 4)


@pytest.mark.parametrize("dtype", DTYPES)
def test_module_falls_back_on_16bit_reference_points(pkg, monkeypatch, dtype):
    """Under autocast with 16-bit reference points the fused entries do not apply: the module takes the unfused path
    and computes exactly what MSDeformAttn(fused=False) computes."""
    torch.manual_seed(1)
    m = pkg.modules.MSDeformAttn(d_model=64, n_levels=2, n_heads=2, n_points=4, fused=True).to(DEV)
    ref_m = pkg.modules.MSDeformAttn(d_model=64, n_levels=2, n_heads=2, n_points=4).to(DEV)
    ref_m.load_state_dict(m.state_dict())
    levels = [(8, 16), (4, 8)]
    shapes, lsi = pkg.synthetic.level_tensors(levels, device=DEV)
    x = torch.randn(1, 160, 64, device=DEV)
    ref = pkg.modules.reference_points_for(levels, DEV).to(dtype)
    calls = []
    fn = pkg.ops.ms_deform_attn_fused_forward
    monkeypatch.setattr(pkg.ops, "ms_deform_attn_fused_forward", lambda *a: calls.append(1) or fn(*a))
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        a, b = m(x, ref, x, shapes, lsi), ref_m(x, ref, x, shapes, lsi)
    assert not calls
    assert torch.equal(a, b)


# ---------------------------------------------------------------- 9. the module and the pixel decoder
@pytest.mark.parametrize("dtype", DTYPES)
def test_module_under_autocast_takes_the_fused_16bit_kernels(pkg, monkeypatch, dtype):
    torch.manual_seed(0)
    kw = dict(d_model=256, n_levels=3, n_heads=8, n_points=4)
    fused = pkg.modules.MSDeformAttn(fused=True, **kw).to(DEV)
    with torch.no_grad():
        for lin in (fused.sampling_offsets, fused.attention_weights):
            torch.nn.init.normal_(lin.weight, std=0.02)
    plain = pkg.modules.MSDeformAttn(**kw).to(DEV)
    plain.load_state_dict(fused.state_dict())
    levels = [(8, 16), (16, 32), (32, 64)]
    shapes, lsi = pkg.synthetic.level_tensors(levels, device=DEV)
    S = sum(h * w for h, w in levels)
    x = torch.randn(2, S, 256, device=DEV)
    ref = pkg.synthetic.reference_points(levels).to(DEV)[None, :, None, :].expand(2, S, 3, 2)
    calls = []
    for name in ("ms_deform_attn_fused_forward", "ms_deform_attn_fused_backward"):
        fn = getattr(pkg.ops, name)
        monkeypatch.setattr(pkg.ops, name, lambda *a, _fn=fn, _n=name: calls.append(_n) or _fn(*a))
    grads = []
    for m in (fused, plain):
        with torch.autocast("cuda", dtype=dtype):
            y = m(x, ref, x, shapes, lsi)
        assert y.dtype == dtype
        # scaled as GradScaler scales an fp16 loss: the 16-bit offset / logit gradients stay out of the subnormal range
        (y.float().square().mean() * 2.0 ** 12).backward()
        grads.append({n: p.grad.float() for n, p in m.named_parameters()})
    assert calls == ["ms_deform_attn_fused_forward", "ms_deform_attn_fused_backward"], calls
    bar = 2.0 ** -8 if dtype == torch.bfloat16 else 2.0 ** -11
    for n, g in grads[0].items():
        assert torch.isfinite(g).all(), n
        r = grads[1][n]
        assert (g - r).norm().item() <= bar * r.norm().item(), f"{n}: {(g - r).norm().item() / r.norm().item()}"


@pytest.mark.parametrize("dtype", DTYPES)
def test_pixel_decoder_amp_fused(pkg, oracle, monkeypatch, dtype):
    """MSDeformAttnPixelDecoder(amp=True, fused=True): forward and training step under autocast on the fused 16-bit
    kernels, within what the composition path moves under a one-ulp perturbation of its inputs."""
    from test_mixed_precision_gpu import _decoder, _nrel, _step, _upcast_oracle_core
    m, feats, _ = _decoder(pkg)
    for mod in m.modules():
        if isinstance(mod, pkg.modules.MSDeformAttn):
            mod.fused = True
    ref_m, _, _ = _decoder(pkg, core=_upcast_oracle_core(oracle))
    gen = torch.Generator().manual_seed(21)
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        mask, low, multi = m.forward_features(feats)
    weights = [torch.randn(o.shape, generator=gen).to(DEV) for o in [mask, low, *multi]]
    calls = []
    for name in ("ms_deform_attn_fused_forward", "ms_deform_attn_fused_backward"):
        fn = getattr(pkg.ops, name)
        monkeypatch.setattr(pkg.ops, name, lambda *a, _fn=fn, _n=name: calls.append(_n) or _fn(*a))
    outs, grads = _step(m, feats, dtype, weights)
    assert "ms_deform_attn_fused_forward" in calls and "ms_deform_attn_fused_backward" in calls, calls
    ref_outs, ref_grads = _step(ref_m, feats, dtype, weights)
    sign = {k: torch.where(torch.rand(v.shape, generator=gen) < 0.5, -1.0, 1.0).to(DEV) for k, v in feats.items()}
    pert = {k: v + sign[k] * torch.from_numpy(ulp16(v.cpu().numpy(), dtype)).float().to(DEV) for k, v in feats.items()}
    p_outs, p_grads = _step(ref_m, pert, dtype, weights)
    assert set(grads) == set(ref_grads)
    for i, (o, r, p) in enumerate(zip(outs, ref_outs, p_outs)):
        assert torch.isfinite(o).all()
        assert _nrel(o, r) <= _nrel(p, r), f"output {i}: {_nrel(o, r)} > {_nrel(p, r)}"
    for n in grads:
        assert torch.isfinite(grads[n]).all(), n
        assert _nrel(grads[n], ref_grads[n]) <= _nrel(p_grads[n], ref_grads[n]), n
