"""The mixed-precision MSDA op (bf16 / fp16 value rows, fp32 locations, weights and sums) and the pixel decoder's
``amp=True`` mode.

Contract: the results equal the fp32 op applied to the widened 16-bit inputs up to ONE rounding of output /
grad_value to the 16-bit type.  So the references are the fp64 oracle on the widened inputs (pure fp64 on
power-of-two pyramids, `f64g32` elsewhere, as test_parity_gpu.py), and the bars are
    forward            |out - ref| <= ulp16(ref) + FWD_ABS_TOL
    grad_value         |d| <= ulp16(ref) + GRAD_REL_TOL * max|ref|
    grad_loc / grad_w  the fp32 GRAD_REL_TOL (their inputs are exact in fp32)
"""
import contextlib

import numpy as np
import pytest
import torch

from conftest import FWD_ABS_TOL, GOLDEN_NAMES, GRAD_REL_TOL, load_golden, rel_err
from test_parity_gpu import _pow2, oracle_refs

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DTYPES = [torch.bfloat16, torch.float16]


def ulp16(x, dtype):
    """One unit in the last place of the 16-bit type at |x| (subnormal spacing below the normal range)."""
    mant, emin = (7, -126) if dtype == torch.bfloat16 else (10, -14)
    a = np.abs(np.asarray(x, dtype=np.float64))
    e = np.floor(np.log2(np.where(a > 0, a, 2.0 ** emin)))
    return 2.0 ** (np.maximum(e, emin) - mant)


def widened(inp, dtype):
    """The inputs with value and grad_output rounded to `dtype` (kept as fp32 CPU tensors: the oracle's view)."""
    out = dict(inp)
    for k in ("value", "grad_output"):
        out[k] = inp[k].to(dtype).float()
    return out


def on_device(inp, dtype):
    return {k: (v.to(dtype) if k in ("value", "grad_output") else v).to(DEV).contiguous() for k, v in inp.items()}


def args_of(d):
    return (d["value"], d["spatial_shapes"], d["level_start_index"], d["sampling_locations"], d["attention_weights"])


def run_mixed(pkg, d):
    out = pkg.ms_deform_attn_mixed_forward(*args_of(d), 128)
    gv, gl, gw = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
    torch.cuda.synchronize()
    return out, gv, gl, gw


def check_mixed(out, gv, gl, gw, refs, dtype, tag="", loc_grad=True):
    ref_out, ref_gv, ref_gl, ref_gw = (np.asarray(r, dtype=np.float64) for r in refs)
    assert out.dtype == dtype and gv.dtype == dtype and gl.dtype == torch.float32 and gw.dtype == torch.float32
    o = out.double().cpu().numpy()
    ref_out = ref_out.reshape(o.shape)
    excess = np.abs(o - ref_out) - (ulp16(ref_out, dtype) + FWD_ABS_TOL)
    assert excess.max() <= 0, f"{tag} forward: {excess.max()}"
    g = gv.double().cpu().numpy()
    ref_gv = ref_gv.reshape(g.shape)
    excess = np.abs(g - ref_gv) - (ulp16(ref_gv, dtype) + GRAD_REL_TOL * np.abs(ref_gv).max())
    assert excess.max() <= 0, f"{tag} grad_value: {excess.max()}"
    assert rel_err(gw.cpu().numpy(), ref_gw) <= GRAD_REL_TOL, f"{tag} grad_attn_weight"
    if loc_grad:
        assert rel_err(gl.cpu().numpy(), ref_gl) <= GRAD_REL_TOL, f"{tag} grad_sampling_loc"


def refs_for(oracle, inp, levels):
    return oracle_refs(oracle, inp, geometry=None if _pow2(levels) else np.float32)


@contextlib.contextmanager
def option(pkg, name, value):
    pkg.set_option(name, value)
    try:
        yield
    finally:
        pkg.set_option(name, 0)


# ---------------------------------------------------------------- accuracy on the op's shapes and paths
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name", GOLDEN_NAMES)
def test_golden_shapes(pkg, oracle, name, dtype):
    g = load_golden(name)
    pinned = bool(g.pop("loc_grad_pinned"))
    inp = widened({k: torch.as_tensor(v) for k, v in g.items() if not k.startswith("ref_")}, dtype)
    levels = [tuple(int(x) for x in hw) for hw in inp["spatial_shapes"].tolist()]
    out, gv, gl, gw = run_mixed(pkg, on_device(inp, dtype))
    check_mixed(out, gv, gl, gw, refs_for(oracle, inp, levels), dtype, tag=name, loc_grad=pinned)


CASES = [
    # levels, batch, heads, channels, points, num_query, mode
    ([(16, 32), (32, 64), (64, 128)], 2, 8, 32, 4, None, "model"),     # merging backward (Lq == S)
    ([(16, 32), (32, 64), (64, 128)], 1, 8, 32, 4, 777, "uniform"),    # Lq != S: per-row backward
    ([(9, 13), (17, 5)], 3, 4, 32, 2, None, "uniform"),                # LP = 4, odd sizes
    ([(7, 9), (5, 3), (4, 4), (2, 2)], 2, 2, 32, 4, None, "uniform"),  # LP = 16
    ([(6, 7), (3, 4)], 2, 3, 32, 3, None, "uniform"),                  # LP = 6 -> generic kernel
    ([(6, 7), (3, 4)], 2, 2, 16, 4, 33, "uniform"),                    # D = 16 -> generic kernel
    ([(6, 7)], 1, 2, 48, 4, 21, "uniform"),                            # D = 48 -> generic kernel
]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("levels,batch,heads,channels,points,nq,mode", CASES)
def test_matches_oracle_on_widened_inputs(pkg, oracle, levels, batch, heads, channels, points, nq, mode, dtype):
    inp = widened(pkg.synthetic.make_inputs(levels, batch, heads, channels, points, num_query=nq, mode=mode,
                                            seed=42), dtype)
    out, gv, gl, gw = run_mixed(pkg, on_device(inp, dtype))
    check_mixed(out, gv, gl, gw, refs_for(oracle, inp, levels), dtype, tag=str(levels))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("name,mode", [("cityscapes_512x1024_b8", "model"), ("cityscapes_512x1024_b8", "uniform"),
                                       ("kitti_384x1248_b16", "model")])
def test_full_size_workloads(pkg, oracle, name, mode, dtype):
    """BASELINE configs[1] (model-like and uniform locations) and the KITTI workload at batch 16."""
    inp = widened(pkg.synthetic.make_workload_inputs(name, mode=mode, seed=3), dtype)
    levels = [tuple(int(x) for x in hw) for hw in inp["spatial_shapes"].tolist()]
    out, gv, gl, gw = run_mixed(pkg, on_device(inp, dtype))
    check_mixed(out, gv, gl, gw, refs_for(oracle, inp, levels), dtype, tag=name)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("mode,bwd_variant", [("model", 2), ("model", 20), ("uniform", 2), ("uniform", 20)])
def test_probe_gated_default_equals_either_backward_kernel(pkg, oracle, mode, bwd_variant, dtype):
    levels = [(16, 32), (32, 64), (64, 128)]
    inp = widened(pkg.synthetic.make_inputs(levels, 1, mode=mode, seed=5), dtype)
    d = on_device(inp, dtype)
    refs = refs_for(oracle, inp, levels)
    out = pkg.ms_deform_attn_mixed_forward(*args_of(d), 128)
    auto = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
    with option(pkg, "bwd_variant", bwd_variant):
        forced = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
    check_mixed(out, *auto, refs, dtype, tag="gated")
    check_mixed(out, *forced, refs, dtype, tag=f"variant {bwd_variant}")


@pytest.mark.parametrize("dtype", DTYPES)
def test_unaligned_value_view(pkg, oracle, dtype):
    """A contiguous view one element into its storage: not 8-byte aligned, the generic kernels serve it."""
    levels = [(16, 32), (32, 64)]
    inp = widened(pkg.synthetic.make_inputs(levels, 2, mode="model", seed=9), dtype)
    d = on_device(inp, dtype)
    for k in ("value", "grad_output"):
        buf = torch.empty(d[k].numel() + 1, dtype=dtype, device=DEV)
        d[k] = buf[1:].view(d[k].shape).copy_(d[k])
    out, gv, gl, gw = run_mixed(pkg, d)
    check_mixed(out, gv, gl, gw, refs_for(oracle, inp, levels), dtype, tag="unaligned")


@pytest.mark.parametrize("dtype", DTYPES)
def test_default_path_runs_the_32_channel_kernels(pkg, oracle, dtype):
    """Launch counts pin the path: forward 1 (the 32-channel kernel; the generic one would also be 1, so the
    forced-generic count below tells them apart only through the backward); backward at Lq == S 3 (merging +
    per-row kernel, both probing, + the conversion), at Lq != S 2 (per-row + conversion).  A value view that is
    16-byte but not 64-byte aligned leaves the merging kernel's row rule unmet and takes the per-row kernel alone."""
    levels = [(16, 32), (32, 64)]
    for nq, expect in ((None, 3), (333, 2)):
        inp = widened(pkg.synthetic.make_inputs(levels, 2, mode="uniform", num_query=nq, seed=4), dtype)
        d = on_device(inp, dtype)
        n0 = pkg.launch_count()
        out = pkg.ms_deform_attn_mixed_forward(*args_of(d), 128)
        assert pkg.launch_count() - n0 == 1
        n0 = pkg.launch_count()
        grads = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
        assert pkg.launch_count() - n0 == expect, nq
        torch.cuda.synchronize()
        check_mixed(out, *grads, refs_for(oracle, inp, levels), dtype, tag=f"default nq={nq}")
    # 16-byte aligned (8 elements in), not 64-byte aligned: per-row kernel + conversion, still exact
    inp = widened(pkg.synthetic.make_inputs(levels, 2, mode="model", seed=6), dtype)
    d = on_device(inp, dtype)
    buf = torch.empty(d["value"].numel() + 8, dtype=dtype, device=DEV)
    d["value"] = buf[8:].view(d["value"].shape).copy_(d["value"])
    assert d["value"].data_ptr() % 16 == 0 and d["value"].data_ptr() % 64 != 0
    out = pkg.ms_deform_attn_mixed_forward(*args_of(d), 128)
    n0 = pkg.launch_count()
    grads = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
    assert pkg.launch_count() - n0 == 2
    with option(pkg, "bwd_variant", 63):            # the generic kernel forced: the same count, other arithmetic path
        generic = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
    torch.cuda.synchronize()
    check_mixed(out, *grads, refs_for(oracle, inp, levels), dtype, tag="16-byte aligned view")
    check_mixed(out, *generic, refs_for(oracle, inp, levels), dtype, tag="generic forced")


# ---------------------------------------------------------------- edge cases
@pytest.mark.parametrize("dtype", DTYPES)
def test_points_off_the_map_and_non_finite_locations(pkg, oracle, dtype):
    levels = [(16, 32), (32, 64)]
    inp = widened(pkg.synthetic.make_inputs(levels, 1, mode="uniform", seed=11), dtype)
    loc = inp["sampling_locations"].clone()
    flat = loc.view(-1, 2)
    bad = torch.arange(0, flat.shape[0], 7)
    specials = torch.tensor([float("nan"), float("inf"), -float("inf"), 1e30, -5.0, 3.0])
    flat[bad, 0] = specials[torch.arange(bad.numel()) % specials.numel()]
    inp["sampling_locations"] = loc
    out, gv, gl, gw = run_mixed(pkg, on_device(inp, dtype))
    for t in (out, gv, gl, gw):
        assert torch.isfinite(t).all()
    check_mixed(out, gv, gl, gw, refs_for(oracle, inp, levels), dtype, tag="off the map")
    assert not gl.view(-1, 2)[bad].any() and not gw.view(-1)[bad].any()


@pytest.mark.parametrize("dtype", DTYPES)
def test_empty_inputs_give_zeros_without_a_launch(pkg, dtype):
    for nq, batch in ((0, 2), (5, 0)):
        inp = pkg.synthetic.make_inputs([(4, 6)], max(batch, 1), heads=2, num_query=nq, mode="uniform")
        d = on_device(inp, dtype)
        if batch == 0:
            d = {k: (v[:0] if k not in ("spatial_shapes", "level_start_index") else v) for k, v in d.items()}
        n0 = pkg.launch_count()
        out = pkg.ms_deform_attn_mixed_forward(*args_of(d), 128)
        grads = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
        assert pkg.launch_count() == n0
        assert out.dtype == dtype and grads[0].dtype == dtype
        for t in (out, *grads):
            assert not t.any()


def test_fp16_grad_value_overflow_is_inf(pkg):
    """Every query samples one pixel: its fp32 grad_value exceeds the fp16 range and must come out as inf (what
    GradScaler looks for), the other pixels as the finite rounded values."""
    levels = [(8, 8)]
    inp = pkg.synthetic.make_inputs(levels, 1, heads=2, points=4, mode="uniform", seed=2)
    inp["sampling_locations"][..., 0] = 4.5 / 8          # pixel (4, 4), exactly on it
    inp["sampling_locations"][..., 1] = 4.5 / 8
    inp["grad_output"] = torch.full_like(inp["grad_output"], 30000.0)
    inp = widened(inp, torch.float16)
    d = on_device(inp, torch.float16)
    gv = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)[0]
    ref = pkg.ms_deform_attn_backward(*(t.float() if t.is_floating_point() else t for t in args_of(d)),
                                      d["grad_output"].float(), 128)[0]
    assert (ref.abs() > 65520).any()
    assert not torch.isnan(gv).any()
    assert torch.equal(torch.isinf(gv), ref.abs() >= 65520)
    fin = ref.abs() < 65504
    assert torch.equal(gv[fin], ref[fin].half())


# ---------------------------------------------------------------- CUDA graphs and deterministic mode
@pytest.mark.parametrize("dtype", DTYPES)
def test_cuda_graph_replays(pkg, dtype):
    inp = widened(pkg.synthetic.make_inputs([(8, 16), (16, 32), (32, 64)], 2, mode="model", seed=5), dtype)
    d = on_device(inp, dtype)
    eager_out = pkg.ms_deform_attn_mixed_forward(*args_of(d), 128)
    eager = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            pkg.ms_deform_attn_mixed_forward(*args_of(d), 128)
            pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gout = pkg.ms_deform_attn_mixed_forward(*args_of(d), 128)
        ggrads = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(gout, eager_out)
        assert torch.equal(ggrads[1], eager[1]) and torch.equal(ggrads[2], eager[2])
        g = ggrads[0].double().cpu().numpy()
        e = eager[0].double().cpu().numpy()
        assert (np.abs(g - e) - (ulp16(e, dtype) + 1e-5 * np.abs(e).max())).max() <= 0


@contextlib.contextmanager
def deterministic_mode():
    was, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn_only)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("levels,batch,heads,channels,points,nq,mode", [CASES[0], CASES[1], CASES[4], CASES[5]])
def test_deterministic_mode(pkg, oracle, monkeypatch, levels, batch, heads, channels, points, nq, mode, dtype):
    """Bit-identical grad_value across calls, graph replays and forced image chunking; the same bar as the
    default path."""
    inp = widened(pkg.synthetic.make_inputs(levels, batch, heads, channels, points, num_query=nq, mode=mode,
                                            seed=13), dtype)
    d = on_device(inp, dtype)
    out = pkg.ms_deform_attn_mixed_forward(*args_of(d), 128)
    with deterministic_mode():
        n0 = pkg.launch_count()
        g1 = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
        assert pkg.launch_count() - n0 == 4           # records, sort, bounds, gather: no accumulation buffer
        g2 = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
        graph = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
        torch.cuda.current_stream().wait_stream(s)
        with torch.cuda.graph(graph):
            gg = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
        graph.replay()
        torch.cuda.synchronize()
        per_image = nq if nq is not None else sum(h * w for h, w in levels)
        monkeypatch.setattr(pkg.ops, "DETERMINISTIC_RECORD_LIMIT", per_image * heads * len(levels) * points * 4)
        g3 = pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"], 128)
    for other in (g2, gg, g3):
        for x, y in zip(g1, other):
            assert torch.equal(x, y)
    check_mixed(out, *g1, refs_for(oracle, inp, levels), dtype, tag="deterministic")


# ---------------------------------------------------------------- the contract at the Python boundary
def test_dtype_contract(pkg):
    inp = pkg.synthetic.make_inputs([(4, 6), (8, 12)], 1, heads=2, points=2, mode="uniform")
    for dtype in DTYPES:
        d = on_device(inp, dtype)
        # the drop-in pair keeps the reference's fp32 / fp64 contract
        with pytest.raises(RuntimeError, match="not implemented for"):
            pkg.ms_deform_attn_forward(*args_of(d), 128)
        with pytest.raises(RuntimeError, match="not implemented for"):
            pkg.ms_deform_attn_backward(*args_of(d), d["grad_output"], 128)
        # 16-bit locations or weights
        for k in ("sampling_locations", "attention_weights"):
            bad = dict(d, **{k: d[k].to(dtype)})
            with pytest.raises(RuntimeError, match="fp32"):
                pkg.ms_deform_attn_mixed_forward(*args_of(bad), 128)
        # mixed 16-bit dtypes
        other = torch.float16 if dtype == torch.bfloat16 else torch.bfloat16
        with pytest.raises(RuntimeError, match="expected scalar type"):
            pkg.ms_deform_attn_mixed_backward(*args_of(d), d["grad_output"].to(other), 128)
        with pytest.raises(RuntimeError, match="batch"):
            pkg.ms_deform_attn_mixed_forward(*args_of(d), 0)
        with pytest.raises(RuntimeError, match="contiguous"):
            pkg.ms_deform_attn_mixed_forward(d["value"].transpose(2, 3), *args_of(d)[1:], 128)
    d = on_device(inp, torch.float32)
    with pytest.raises(RuntimeError, match="not implemented for"):
        pkg.ms_deform_attn_mixed_forward(*args_of(d), 128)
    with pytest.raises(RuntimeError, match="CPU"):
        pkg.ms_deform_attn_mixed_forward(*(t.cpu() for t in args_of(on_device(inp, torch.bfloat16))), 128)


@pytest.mark.parametrize("dtype", DTYPES)
def test_module_under_autocast_reaches_the_16bit_entries(pkg, dtype):
    torch.manual_seed(0)
    m = pkg.modules.MSDeformAttn(d_model=256, n_levels=3, n_heads=8, n_points=4, fused=True).to(DEV)
    levels = [(8, 16), (16, 32), (32, 64)]
    shapes, lsi = pkg.synthetic.level_tensors(levels, device=DEV)
    S = sum(h * w for h, w in levels)
    x = torch.randn(2, S, 256, device=DEV, requires_grad=True)
    ref = pkg.synthetic.reference_points(levels).to(DEV)[None, :, None, :].expand(2, S, 3, 2)
    timing = pkg.ops.enable_timing(True)
    try:
        with torch.autocast("cuda", dtype=dtype):
            y = m(x, ref, x, shapes, lsi)
        y.float().square().mean().backward()
        kinds = [k for k, _, _ in timing]
    finally:
        pkg.ops.enable_timing(False)
    assert y.dtype == dtype
    assert kinds == ["forward_mixed", "backward_mixed"], kinds
    assert torch.isfinite(x.grad).all() and x.grad.abs().sum() > 0
    assert all(torch.isfinite(p.grad).all() for p in m.parameters())


# ---------------------------------------------------------------- the pixel decoder under autocast
def _decoder(pkg, core=None, amp=True, linear="torch"):
    from test_pixel_decoder import build
    return build(pkg, core=core, device=DEV, linear=linear) if not amp else _amp_build(pkg, core, linear)


def _amp_build(pkg, core, linear):
    from test_pixel_decoder import PD_KW, PD_SHAPES
    g = load_golden("pixel_decoder_small")
    m = pkg.pixel_decoder.MSDeformAttnPixelDecoder(PD_SHAPES, core=core, linear=linear, amp=True, **PD_KW)
    state = {k[len("state::"):]: torch.from_numpy(v) for k, v in g.items() if k.startswith("state::")}
    m.load_state_dict(state, strict=True)
    feats = {k[len("feat::"):]: torch.from_numpy(v).to(DEV) for k, v in g.items() if k.startswith("feat::")}
    return m.to(DEV).eval(), feats, g


def _upcast_oracle_core(oracle):
    def core(value, shapes, lsi, loc, w, im2col_step):
        return oracle.core_grid_sample(value.float(), shapes, loc.float(), w.float()).to(value.dtype)
    return core


def _step(m, feats, dtype, weights):
    """forward_features under autocast, then the backward of a fixed random projection of its outputs ->
    (outputs, parameter gradients) as fp32."""
    m.zero_grad(set_to_none=True)
    with torch.autocast("cuda", dtype=dtype):
        mask, low, multi = m.forward_features(feats)
    outs = [mask, low] + list(multi)
    loss = sum((o.float() * w).sum() for o, w in zip(outs, weights))
    loss.backward()
    grads = {n: p.grad.float().clone() for n, p in m.named_parameters() if p.grad is not None}
    return [o.detach().float() for o in outs], grads


def _nrel(a, b):
    den = b.norm().item()
    return (a - b).norm().item() / den if den > 0 else (a - b).norm().item()


@pytest.mark.parametrize("dtype", DTYPES)
def test_pixel_decoder_forward_and_training_step_under_autocast(pkg, oracle, dtype):
    m, feats, _ = _decoder(pkg)
    ref_m, _, _ = _decoder(pkg, core=_upcast_oracle_core(oracle))
    gen = torch.Generator().manual_seed(21)
    with torch.no_grad(), torch.autocast("cuda", dtype=dtype):
        mask, low, multi = m.forward_features(feats)
    shapes = [o.shape for o in [mask, low, *multi]]
    weights = [torch.randn(s, generator=gen).to(DEV) for s in shapes]
    n0 = pkg.launch_count()
    outs, grads = _step(m, feats, dtype, weights)
    assert pkg.launch_count() > n0                      # the library's mixed kernels ran
    ref_outs, ref_grads = _step(ref_m, feats, dtype, weights)
    # the bar: what the composition path itself moves when every input feature moves by one 16-bit ulp
    sign = {k: torch.where(torch.rand(v.shape, generator=gen) < 0.5, -1.0, 1.0).to(DEV) for k, v in feats.items()}
    pert = {k: v + sign[k] * torch.from_numpy(ulp16(v.cpu().numpy(), dtype)).float().to(DEV) for k, v in feats.items()}
    p_outs, p_grads = _step(ref_m, pert, dtype, weights)
    assert set(grads) == set(ref_grads)
    for i, (o, r, p) in enumerate(zip(outs, ref_outs, p_outs)):
        assert torch.isfinite(o).all()
        assert _nrel(o, r) <= _nrel(p, r), f"output {i}: {_nrel(o, r)} > {_nrel(p, r)}"
    for n in grads:
        assert torch.isfinite(grads[n]).all(), n
        assert _nrel(grads[n], ref_grads[n]) <= _nrel(p_grads[n], ref_grads[n]), \
            f"{n}: {_nrel(grads[n], ref_grads[n])} > {_nrel(p_grads[n], ref_grads[n])}"


def test_pixel_decoder_amp_defaults_are_unchanged(pkg):
    plain, feats, _ = _decoder(pkg, amp=False)
    amp, _, _ = _decoder(pkg, amp=True)
    with torch.no_grad():
        ref = plain.forward_features(feats)
        no_autocast = amp.forward_features(feats)                  # amp=True, no autocast active
        with torch.autocast("cuda", dtype=torch.bfloat16):
            enclosed = plain.forward_features(feats)               # amp=False inside an autocast
    for a, b, c in zip([ref[0], ref[1], *ref[2]], [no_autocast[0], no_autocast[1], *no_autocast[2]],
                       [enclosed[0], enclosed[1], *enclosed[2]]):
        assert torch.equal(a, b) and torch.equal(a, c)


def test_pixel_decoder_amp_with_tf32x3_raises(pkg):
    from test_pixel_decoder import PD_KW, PD_SHAPES
    with pytest.raises(ValueError, match="tf32x3"):
        pkg.pixel_decoder.MSDeformAttnPixelDecoder(PD_SHAPES, linear="tf32x3", amp=True, **PD_KW)
