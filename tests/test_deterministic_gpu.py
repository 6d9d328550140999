"""GPU tests of the deterministic mode: with torch.use_deterministic_algorithms(True) every backward of the library
(the MSDA op plain and fused, the weight gradient, the residual + LayerNorm backward) and the split-K forward of the
tensor-core Linear give bit-identical results for bit-identical inputs, still meet the accuracy bars of the default
entries, and whole training steps repeat bit for bit."""
import contextlib
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import GRAD_REL_TOL, rel_err
from test_fused_gpu import make_case, reference_composition
from test_linear_gpu import ERR_FACTOR
from test_parity_gpu import _pow2, check_against, oracle_refs, to_dev

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@contextlib.contextmanager
def deterministic_mode(on=True):
    was, warn_only = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(on)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(was, warn_only=warn_only)


@pytest.fixture
def det():
    with deterministic_mode():
        yield


def _in_fresh_process(call):
    """`call` (a call of a function of this module, as source) in a new Python process whose environment has
    CUBLAS_WORKSPACE_CONFIG=:4096:8 (when unset) from its start -> what it returns, as text.  torch's own cuBLAS GEMMs
    are reproducible in deterministic mode only with that setting, and torch fixes the cuBLAS workspace at the
    first GEMM of a process: set here, in this one, it would change the cuBLAS kernels (and the fp32 reference
    errors) of every other test module."""
    code = (f"import sys; sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]\n"
            f"import test_deterministic_gpu as t\nprint(t.{call})")
    env = dict(os.environ)
    env.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    args = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    res = subprocess.run(args, env=env, capture_output=True, text=True, timeout=1200)
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-4000:]
    return res.stdout.strip().splitlines()[-1]


def _flag_off(fn):
    """torch's own reference computations (fp32 / fp64 GEMMs) with the flag off, as in the default entries' tests."""
    with deterministic_mode(False):
        return fn()


def _equal(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


def _no_nan(ts):
    return all(not torch.isnan(t).any().item() for t in ts)


def _graph_replays(fn):
    """fn() captured into a CUDA graph and replayed twice -> (outputs after replay 1, after replay 2)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = fn()
    graph.replay()
    first = [t.clone() for t in outs]
    graph.replay()
    torch.cuda.synchronize()
    return first, [t.clone() for t in outs]


def _records_per_image(t_loc):
    N, Lq, M, L, P, _ = t_loc.shape
    return Lq * M * L * P * 4


# ---------------------------------------------------------------- 1. the MSDA op
OP_CASES = [("cityscapes_512x1024_b8", "model", None), ("cityscapes_512x1024_b8", "uniform", None),
            ("kitti_384x1248_b16", "model", 3)]      # KITTI: L*P = 12, sizes that are not powers of two


@pytest.mark.parametrize("name,mode,batch", OP_CASES)
def test_plain_backward_is_reproducible_and_accurate(pkg, oracle, det, monkeypatch, name, mode, batch):
    inp = pkg.synthetic.make_workload_inputs(name, mode=mode, seed=3, batch=batch)
    d = to_dev(inp)
    a = (d["value"], d["spatial_shapes"], d["level_start_index"], d["sampling_locations"], d["attention_weights"])
    bwd = lambda *t: pkg.ms_deform_attn_backward(*t, 128)                       # noqa: E731
    g1 = bwd(*a, d["grad_output"])
    g2 = bwd(*a, d["grad_output"])
    assert _no_nan(g1) and _equal(g1, g2)
    r1, r2 = _graph_replays(lambda: bwd(*a, d["grad_output"]))
    assert _equal(r1, g1) and _equal(r2, g1)
    N = d["value"].size(0)
    for n in range(N):                                   # each image alone == its rows of the batch call
        one = bwd(*(t[n:n + 1] if i in (0, 3, 4) else t for i, t in enumerate(a)), d["grad_output"][n:n + 1])
        assert all(torch.equal(o[0], g[n]) for o, g in zip(one, g1)), n
    monkeypatch.setattr(pkg.ops, "DETERMINISTIC_RECORD_LIMIT", 2 * _records_per_image(d["sampling_locations"]) + 1)
    assert _equal(bwd(*a, d["grad_output"]), g1)        # chunks of two images
    out = pkg.ms_deform_attn_forward(*a, 128)
    levels = pkg.synthetic.WORKLOADS[name].levels
    ia = (inp["value"], inp["spatial_shapes"], inp["level_start_index"], inp["sampling_locations"],
          inp["attention_weights"])
    if _pow2(levels):
        check_against(out, *g1, oracle.forward(*ia), *oracle.backward(inp["grad_output"], *ia), tag=name + " fp64")
    else:
        check_against(out, *g1, *oracle_refs(oracle, inp), tag=name + " f64g32")


@pytest.mark.parametrize("levels,batch,shared_ref", [
    ([(16, 32), (32, 64), (64, 128)], 8, True),        # configs[1] pyramid and batch
    ([(12, 39), (24, 78), (48, 156)], 3, False),       # KITTI pyramid, per-image reference points
])
def test_fused_backward_is_reproducible_and_accurate(pkg, oracle, det, monkeypatch, levels, batch, shared_ref):
    c = make_case(pkg, levels, batch, 8, 4, shared_ref, seed=23)
    d = {k: (v.to(DEV) if torch.is_tensor(v) else v) for k, v in c.items()}
    a = (d["value"], d["shapes"], d["lsi"], d["ref"], d["off"], d["logits"])
    bwd = lambda *t: pkg.ms_deform_attn_fused_backward(*t)                      # noqa: E731
    g1 = bwd(*a, d["grad_out"])
    assert _no_nan(g1) and _equal(g1, bwd(*a, d["grad_out"]))
    r1, r2 = _graph_replays(lambda: bwd(*a, d["grad_out"]))
    assert _equal(r1, g1) and _equal(r2, g1)
    for n in range(batch):
        ref_n = d["ref"] if shared_ref else d["ref"][n:n + 1]
        one = bwd(d["value"][n:n + 1], d["shapes"], d["lsi"], ref_n, d["off"][n:n + 1], d["logits"][n:n + 1],
                  d["grad_out"][n:n + 1])
        assert all(torch.equal(o[0], g[n]) for o, g in zip(one, g1)), n
    monkeypatch.setattr(pkg.ops, "DETERMINISTIC_RECORD_LIMIT", 2 * _records_per_image(d["off"]) + 1)
    assert _equal(bwd(*a, d["grad_out"]), g1)
    _, ref_gv, ref_goff, ref_glog = reference_composition(oracle, c)
    assert rel_err(g1[0].cpu().numpy(), ref_gv.reshape(g1[0].shape)) <= GRAD_REL_TOL
    assert rel_err(g1[1].cpu().numpy(), ref_goff) <= GRAD_REL_TOL
    assert rel_err(g1[2].cpu().numpy(), ref_glog) <= GRAD_REL_TOL


# ---------------------------------------------------------------- 2. edge cases
@pytest.mark.parametrize("levels,batch,heads,channels,points,nq,dtype,variant", [
    ([(6, 7), (3, 4)], 2, 2, 64, 4, 33, torch.float32, 0),     # D = 64: generic kernel
    ([(6, 7), (3, 4)], 2, 3, 32, 3, None, torch.float32, 0),   # L*P = 6: generic kernel
    ([(9, 13), (17, 5)], 2, 4, 32, 2, None, torch.float32, 63),  # fast-path shape forced onto the generic kernel
    ([(6, 7), (3, 4)], 2, 2, 48, 4, 21, torch.float64, 0),     # fp64
])
def test_generic_kernels(pkg, oracle, det, levels, batch, heads, channels, points, nq, dtype, variant):
    inp = pkg.synthetic.make_inputs(levels, batch, heads, channels, points, num_query=nq, mode="uniform", seed=5)
    d = to_dev(inp, dtype=dtype)
    a = (d["value"], d["spatial_shapes"], d["level_start_index"], d["sampling_locations"], d["attention_weights"])
    pkg.set_option("bwd_variant", variant)
    try:
        g1 = pkg.ms_deform_attn_backward(*a, d["grad_output"], 128)
        g2 = pkg.ms_deform_attn_backward(*a, d["grad_output"], 128)
    finally:
        pkg.set_option("bwd_variant", 0)
    assert _no_nan(g1) and _equal(g1, g2)
    out = pkg.ms_deform_attn_forward(*a, 128)
    if dtype == torch.float64:          # pure fp64 oracle
        ia = (inp["value"], inp["spatial_shapes"], inp["level_start_index"], inp["sampling_locations"],
              inp["attention_weights"])
        rgv, _, rgw = oracle.backward(inp["grad_output"], *ia)
        assert rel_err(g1[0].cpu().numpy(), np.reshape(rgv, g1[0].shape)) <= 1e-10
        assert rel_err(g1[2].cpu().numpy(), rgw) <= 1e-10
    else:
        check_against(out, *g1, *oracle_refs(oracle, inp), tag=str(levels))


def test_fp64_gradcheck(pkg, det):
    inp = pkg.synthetic.make_inputs([(3, 4), (2, 3)], 1, 2, 3, 2, num_query=3, mode="uniform", seed=6,
                                    dtype=torch.float64)
    d = to_dev(inp, dtype=torch.float64)
    value = d["value"].clone().requires_grad_(True)
    loc = d["sampling_locations"].clone().requires_grad_(True)
    w = d["attention_weights"].clone().requires_grad_(True)
    f = lambda v, lo, ww: pkg.MSDeformAttnFunction.apply(v, d["spatial_shapes"], d["level_start_index"], lo, ww, 2)  # noqa: E731
    assert torch.autograd.gradcheck(f, (value, loc, w), eps=1e-6, atol=1e-5, nondet_tol=0.0)


def test_locations_outside_the_map_and_non_finite(pkg, det):
    inp = pkg.synthetic.make_inputs([(16, 32), (8, 16)], 2, 4, 32, 4, mode="uniform", seed=7)
    d = to_dev(inp)
    loc = d["sampling_locations"].clone()
    flat = loc.view(-1, 2)
    g = torch.Generator(device=DEV).manual_seed(1)
    pick = torch.randint(0, flat.size(0), (flat.size(0) // 3,), device=DEV, generator=g)
    bad = torch.tensor([[-5.0, 0.5], [0.5, 3.0], [float("nan"), 0.5], [0.5, float("inf")], [-0.01, -0.01],
                        [1.01, 0.99]], device=DEV)
    flat[pick] = bad[torch.arange(pick.numel(), device=DEV) % bad.size(0)]
    a = (d["value"], d["spatial_shapes"], d["level_start_index"], loc, d["attention_weights"])
    g1 = pkg.ms_deform_attn_backward(*a, d["grad_output"], 128)
    assert _no_nan(g1) and _equal(g1, pkg.ms_deform_attn_backward(*a, d["grad_output"], 128))
    torch.use_deterministic_algorithms(False)
    g0 = pkg.ms_deform_attn_backward(*a, d["grad_output"], 128)
    torch.use_deterministic_algorithms(True)
    assert torch.equal(g1[1], g0[1]) and torch.equal(g1[2], g0[2])       # computed exactly as by the default
    assert rel_err(g1[0].cpu().numpy(), g0[0].cpu().numpy()) <= 1e-5


def test_every_sample_on_one_pixel(pkg, det):
    """All 131 072 samples of 32 768 queries at the centre of one pixel: one bucket of 131 072 records (corner 0),
    three buckets of zero-weight records, every other row empty."""
    levels, Lq, P = [(8, 8)], 32768, 4
    shapes, lsi = pkg.synthetic.level_tensors(levels, DEV)
    g = torch.Generator(device=DEV).manual_seed(2)
    value = torch.randn(1, 64, 1, 32, device=DEV, generator=g)
    loc = torch.empty(1, Lq, 1, 1, P, 2, device=DEV)
    loc[..., 0], loc[..., 1] = (3 + 0.5) / 8, (5 + 0.5) / 8                  # pixel (x=3, y=5)
    w = torch.rand(1, Lq, 1, 1, P, device=DEV, generator=g)
    go = torch.randn(1, Lq, 32, device=DEV, generator=g)
    gv, gl, gw = pkg.ms_deform_attn_backward(value, shapes, lsi, loc, w, go, 128)
    assert _equal((gv, gl, gw), pkg.ms_deform_attn_backward(value, shapes, lsi, loc, w, go, 128))
    want = torch.zeros(64, 32, dtype=torch.float64, device=DEV)
    want[5 * 8 + 3] = (w.double().sum(-1).view(Lq, 1) * go.double().view(Lq, 32)).sum(0)
    got = gv.view(64, 32).double()
    assert ((got - want).abs().max() / want.abs().max()).item() <= 1e-4      # a sequential fp32 sum of 131 072 terms
    assert not got[torch.arange(64, device=DEV) != 5 * 8 + 3].any().item()


# ---------------------------------------------------------------- 3. Linear layers and LayerNorm
def test_linear_wgrad(pkg, det):
    g = torch.Generator().manual_seed(11)
    rows, out_f, in_f = 5000, 256, 256                  # 9 chunks of 512 rows and a ragged tenth
    gy = torch.randn(rows, out_f, generator=g).to(DEV)
    x = torch.randn(rows, in_f, generator=g).to(DEV)
    gw, gb = pkg.ops.linear_wgrad(gy, x)
    assert _equal((gw, gb), pkg.ops.linear_wgrad(gy, x))
    ref, y32 = _flag_off(lambda: (gy.double().t() @ x.double(), gy.t() @ x))
    err, err32 = (gw.double() - ref).abs().max().item(), (y32.double() - ref).abs().max().item()
    assert err <= ERR_FACTOR * err32 + 2e-6 * ref.abs().max().item(), (err, err32)
    refb = gy.double().sum(0)
    assert (gb.double() - refb).abs().max().item() <= 4 * (gy.sum(0).double() - refb).abs().max().item() + 1e-4
    gw2, none = pkg.ops.linear_wgrad(gy, x, with_bias=False)
    assert none is None and torch.equal(gw2, gw)


def test_linear_split_k_shape(pkg, det):
    g = torch.Generator().manual_seed(12)
    x = torch.randn(256, 4096, generator=g).to(DEV)
    w = torch.randn(256, 4096, generator=g).to(DEV)
    y = pkg.linear_tf32x3(x, w, None, split_weight_in_kernel=True)      # split-K when the flag is off
    assert torch.equal(y, pkg.linear_tf32x3(x, w, None, split_weight_in_kernel=True))
    ref, y32 = _flag_off(lambda: (x.double() @ w.double().t(), x @ w.t()))
    err, err32 = (y.double() - ref).abs().max().item(), (y32.double() - ref).abs().max().item()
    assert err <= ERR_FACTOR * err32 + 1e-6, (err, err32)
    # outside split-K shapes the deterministic entries are the default ones
    xs, ws, b = x[:, :256].contiguous(), w[:, :256].contiguous(), torch.randn(256, generator=g).to(DEV)
    on = [pkg.linear_tf32x3(xs, ws, b), pkg.linear_tf32x3(xs, ws, b, presplit=pkg.ops.split_weight(ws))]
    torch.use_deterministic_algorithms(False)
    off = [pkg.linear_tf32x3(xs, ws, b), pkg.linear_tf32x3(xs, ws, b, presplit=pkg.ops.split_weight(ws))]
    torch.use_deterministic_algorithms(True)
    assert _equal(on, off)


@pytest.mark.parametrize("rows,cols", [(77, 128), (344064, 256)])
def test_add_layernorm_backward(pkg, det, rows, cols):
    g = torch.Generator().manual_seed(rows)
    x = (torch.randn(rows, cols, generator=g) * 2 + 0.5).to(DEV)
    r = torch.randn(rows, cols, generator=g).to(DEV)
    w = (torch.randn(cols, generator=g) + 1).to(DEV)
    cot = torch.randn(rows, cols, generator=g).to(DEV)
    got = pkg.ops.add_layernorm_backward(cot, x, r, w, 1e-5)
    assert _equal(got, pkg.ops.add_layernorm_backward(cot, x, r, w, 1e-5))
    torch.use_deterministic_algorithms(False)
    assert torch.equal(pkg.ops.add_layernorm_backward(cot, x, r, w, 1e-5)[0], got[0])
    ref = [t.clone().double().requires_grad_(True) for t in (x, r, w)]
    b64 = torch.zeros(cols, dtype=torch.float64, device=DEV, requires_grad=True)
    (F.layer_norm(ref[0] + ref[1], (cols,), ref[2], b64, 1e-5) * cot.double()).sum().backward()
    t32 = [t.clone().requires_grad_(True) for t in (x, r, w)]
    b32 = torch.zeros(cols, device=DEV, requires_grad=True)
    (F.layer_norm(t32[0] + t32[1], (cols,), t32[2], b32, 1e-5) * cot).sum().backward()
    torch.use_deterministic_algorithms(True)
    for mine, r64, r32 in zip(got, (ref[0].grad, ref[2].grad, b64.grad), (t32[0].grad, t32[2].grad, b32.grad)):
        err, err32 = (mine.double() - r64).abs().max().item(), (r32.double() - r64).abs().max().item()
        assert err <= 3 * err32 + 1e-6 * max(1.0, r64.abs().max().item()), (err, err32)


# ---------------------------------------------------------------- 4./5. whole training steps
def _encoder(pkg, fused, linear):
    torch.manual_seed(0)
    m = pkg.modules.MSDeformAttnTransformerEncoderOnly(
        d_model=256, nhead=8, num_encoder_layers=2, dim_feedforward=1024, dropout=0.1, num_feature_levels=3,
        enc_n_points=4, fused=fused, linear=linear).to(DEV).train()
    with torch.no_grad():                                  # small learned offsets, as in a trained model
        for layer in m.encoder.layers:
            torch.nn.init.normal_(layer.self_attn.sampling_offsets.weight, std=0.02)
            torch.nn.init.normal_(layer.self_attn.attention_weights.weight, std=0.05)
    g = torch.Generator(device=DEV).manual_seed(1)
    levels = pkg.synthetic.pyramid(256, 512)
    srcs = [torch.randn(2, 256, h, w, device=DEV, generator=g) for h, w in levels]
    pos = [torch.randn(2, 256, h, w, device=DEV, generator=g) * 0.1 for h, w in levels]
    return m, (srcs, pos)


def _decoder(pkg):
    torch.manual_seed(5)
    shapes = {"res2": (96, 4), "res3": (192, 8), "res4": (384, 16), "res5": (768, 32)}
    m = pkg.pixel_decoder.MSDeformAttnPixelDecoder(
        shapes, transformer_dropout=0.1, transformer_nheads=8, transformer_dim_feedforward=1024,
        transformer_enc_layers=2, conv_dim=256, mask_dim=256, norm="GN", transformer_in_features=["res3", "res4", "res5"],
        common_stride=4, fused=True, linear="tf32x3").to(DEV).train()
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, pkg.modules.MSDeformAttn):
                torch.nn.init.normal_(mod.sampling_offsets.weight, std=0.02)
                torch.nn.init.normal_(mod.attention_weights.weight, std=0.05)
    g = torch.Generator(device=DEV).manual_seed(6)
    feats = {k: torch.randn(2, c, 128 // s, 256 // s, device=DEV, generator=g) for k, (c, s) in shapes.items()}
    return m, feats


def _step(m, state, run):
    """Load `state`, then one seeded step: forward (dropout 0.1) -> loss -> backward -> AdamW.
    -> (loss, outputs, gradients of every parameter and input, parameters after the step)."""
    m.load_state_dict(state)
    opt = torch.optim.AdamW(m.parameters(), lr=1e-3)
    opt.zero_grad(set_to_none=True)
    torch.manual_seed(123)
    outs, leaves = run()
    loss = sum(o.square().mean() for o in outs)
    loss.backward()
    grads = {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}
    grads.update({f"input{i}": t.grad.clone() for i, t in enumerate(leaves)})
    opt.step()
    return loss.detach(), [o.detach() for o in outs], grads, {n: p.detach().clone() for n, p in m.named_parameters()}


def _encoder_run(m, inputs):
    def run():
        srcs = [t.clone().requires_grad_(True) for t in inputs[0]]
        pos = [t.clone() for t in inputs[1]]
        return [m(srcs, pos)[0]], srcs
    return run


def _decoder_run(m, feats):
    def run():
        leaves = {k: v.clone().requires_grad_(True) for k, v in feats.items()}
        mask, low, multi = m.forward_features(leaves)
        return [mask, low, *multi], list(leaves.values())
    return run


def _repeat_twice(m, run):
    state = {k: v.clone() for k, v in m.state_dict().items()}
    flags = torch.backends.cudnn.deterministic, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        a, b = _step(m, state, run), _step(m, state, run)
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = flags
    return state, a, b


def _assert_same_step(a, b):
    assert torch.equal(a[0], b[0])
    assert _equal(a[1], b[1])
    assert set(a[2]) == set(b[2]) and all(torch.equal(a[2][k], b[2][k]) for k in a[2]), \
        [k for k in a[2] if not torch.equal(a[2][k], b[2][k])]
    assert all(torch.equal(a[3][k], b[3][k]) for k in a[3])


def _load():
    from __graft_entry__ import load_package
    return load_package()


def encoder_step_twice(fused, linear):
    pkg = _load()
    m, inputs = _encoder(pkg, fused, linear)
    with deterministic_mode():
        _, a, b = _repeat_twice(m, _encoder_run(m, inputs))
    _assert_same_step(a, b)
    return "same"


def decoder_step_twice():
    pkg = _load()
    m, feats = _decoder(pkg)
    with deterministic_mode():
        _, a, b = _repeat_twice(m, _decoder_run(m, feats))
    _assert_same_step(a, b)
    return "same"


def encoder_step_flag_on_and_off():
    """-> the worst per-tensor gradient difference (norm-relative) of the step with the flag on against off."""
    pkg = _load()
    m, inputs = _encoder(pkg, True, "tf32x3")
    with deterministic_mode():
        state, on, _ = _repeat_twice(m, _encoder_run(m, inputs))
    m.load_state_dict(state)
    _, off, _ = _repeat_twice(m, _encoder_run(m, inputs))
    assert _equal(on[1], off[1])

    def rel(x, y):
        return ((x.double() - y.double()).norm() / y.double().norm().clamp_min(1e-30)).item()
    err = {k: rel(on[2][k], off[2][k]) for k in off[2]}
    worst = max(err.items(), key=lambda kv: kv[1])
    return f"{worst[1]!r} {worst[0]}"


@pytest.mark.parametrize("fused,linear", [(True, "tf32x3"), (False, "torch")])
def test_encoder_training_step_repeats_bit_for_bit(fused, linear):
    assert _in_fresh_process(f"encoder_step_twice({fused!r}, {linear!r})") == "same"


def test_pixel_decoder_training_step_repeats_bit_for_bit():
    assert _in_fresh_process("decoder_step_twice()") == "same"


def test_flag_on_and_off_differ_only_by_rounding():
    """The same encoder step (fused producers, tensor-core linears) with the flag on and off: identical forward
    outputs, gradients within rounding of each other (per tensor, norm-relative)."""
    worst, name = _in_fresh_process("encoder_step_flag_on_and_off()").split()
    print(f"\nencoder step, flag on against off: worst per-tensor gradient difference {float(worst):.3g} ({name})")
    assert float(worst) <= 1e-5, (worst, name)
