"""Mixed-precision MSDA on the B200: the bf16 / fp16 op against fp32, and the pixel decoder under autocast.

    python tools/bench_mixed.py [--parts a,b,c] [--steps 20] [--out DIR]

DIR defaults to $BENCH_OUT/mixed, and BENCH_OUT to bench_out/ in the repository (git-ignored).

(a) the op alone at BASELINE configs[1] (512x1024, batch 8) and at the configs[2] shape (1024x2048, batch 8):
    forward, backward (gated default, merging kernel forced, per-row kernel forced) and forward + backward, for
    fp32, bf16 and fp16 on the same seeded inputs (value / grad_output rounded once to the 16-bit type), the three
    types alternating in one process.  Every timed call follows a 256 MB write that evicts the 126 MB L2; the
    events bracket the call only.  Times are of the Python-level call, so the 16-bit backward includes the
    zero-fill of its fp32 accumulation buffer (torch) and the conversion launch.  Algorithmic bytes from shapes:
    value / output / grad_output / grad_value once each at their element size, locations and weights (12 bytes a
    point) and their gradients once -- per query at configs[1] 3 200 (fp32) / 2 176 (16-bit) forward and
    5 376 / 3 840 backward; the accumulation buffer's zero-fill and conversion read (4 + 4 bytes per value
    element) are reported separately.
(f) part (a)'s fused-producer arms at the same two shapes (raw offsets [N, Lq, M, L, P, 2] and logits [N, Lq, M, L*P]
    as the Linear layers hand them over, fp32 reference points): per 16-bit type the fused 16-bit op against the
    unfused 16-bit composition MSDeformAttn(fused=False) runs under autocast (torch's fp32 softmax and
    `ref + off.float() / (W, H)`, then the mixed-precision op) and against the fp32 fused op; forward, backward and
    both, through autograd (the backward arm's forward runs untimed just before it), arms alternating and the L2
    evicted before every timed call as in (a).
(b) the decoder forward (forward_features, no autograd) at the configs[2] shape with a Swin-T pyramid: the fastest
    fp32 setting (fused=True, linear="tf32x3") against amp=True under bf16 autocast, with fused=True (the fused 16-bit
    kernels) and fused=False (torch's producers around the mixed-precision op).
(c) the decoder training step (forward_features -> loss -> backward -> AdamW) at 512x1024, batch 16, as
    tools/bench_decoder_train.py: fp32 linear="tf32x3" against amp=True with bf16, and with fp16 + GradScaler, each
    with fused=True and fused=False.

(l) the residual + LayerNorm site of the encoder alone at 344 064 x 256 (configs[2]'s rows), bf16 and fp16, forward and
    backward: the mixed-precision kernels (fp32 x, 16-bit residual -> fp32 y and its 16-bit copy; backward from both
    gradients) against torch's autocast composition of the same site (add, layer_norm, the cast for the next GEMM;
    autograd for the backward) and against the fp32 kernels (fp32 residual, no copy).  Arms alternate, the L2 is
    evicted before every call.  Algorithmic bytes per element: forward 4 + 2 in, 4 + 2 out; backward 4 + 2 + 4 + 2 in,
    4 + 2 out (fp32 kernels: 4 + 4 in, 4 out; 4 + 4 + 4 in, 4 out), and their share of the measured HBM figure.
(p) the 16-bit packed / per-query-table forward (one [N, Lq, 3*M*L*P] projection output and the fp32 table) against
    the 16-bit fused forward on separate offset / logit tensors and the fp32 packed forward with the table, at
    configs[1] and the configs[2] shape; arms alternate, L2 evicted before every call.
(g) the decoder's GroupNorm sites at the configs[2] shape (1024x2048, batch 8, Swin-T, conv_dim 256), bf16 and fp16:
    the FPN lateral (GroupNorm + the up-sampled fp32 encoder level, [8, 256, 256, 512] with up [8, 256, 128, 256]) and
    output (GroupNorm + ReLU) maps, both returning the 16-bit copy, and the three input projections written as fp32
    rows of one [8, S, 256] tensor (with the convolution bias added on the fly); forward and backward (from the 16-bit
    gradient for the two FPN maps, the fp32 rows gradient for the projections).  Arms: the 16-bit kernels, torch's
    autocast composition (autograd for the backward; its forward runs untimed just before), and the fp32 kernels on
    the widened map.  Arms alternate, the L2 is evicted before every call.  Algorithmic bytes per element of the map
    (16-bit kernels): forward 2 + 2 read, 2 written (rows: 4 written), + 4 per element of `up`; backward 2 + 2 + 2 + 2
    read, 2 written (rows: 4 + 2 + 4 + 2 read), + 2 read and 4 written per element of `up` for its gradient; the fp32
    kernels 4 for every 2.  Torch's arm is charged the 16-bit kernels' bytes (the site's minimum).
Parts (b) and (c) carry linear="autocast" arms next to the others, and the linear="autocast" arms with the 16-bit
GroupNorm kernels off (the predicates patched to refuse 16-bit maps); the arms of (b) and (c) alternate.

Every JSON line carries the card's name and power limit (read-only nvidia-smi query).
"""
import argparse
import contextlib
import json
import os
import statistics
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from __graft_entry__ import load_package  # noqa: E402
from bench_decoder_train import card, timed  # noqa: E402

DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}
HBM_GBS = 6540.8          # the project's measured HBM bandwidth on the B200 (DESIGN.md section 10)
SWIN_T = {"res2": (96, 4), "res3": (192, 8), "res4": (384, 16), "res5": (768, 32)}


def op_bytes(inp, esize):
    N, S, M, D = inp["value"].shape
    Lq, L, P = inp["sampling_locations"].shape[1], inp["sampling_locations"].shape[3], inp["sampling_locations"].shape[4]
    rows_v, rows_q, pts = N * S * M * D, N * Lq * M * D, N * Lq * M * L * P
    return {"forward": rows_v * esize + rows_q * esize + pts * 12,
            "backward": 2 * rows_v * esize + rows_q * esize + 2 * pts * 12,
            "accum_zero_fill": rows_v * 4 if esize == 2 else 0, "accum_conversion_read": rows_v * 4 if esize == 2 else 0,
            "queries": N * Lq}


def part_a(pkg, args, emit):
    dev = torch.device("cuda", 0)
    dtypes = {k: DTYPES[k] for k in args.dtypes.split(",")}
    ops = args.ops.split(",")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for name in ("cityscapes_512x1024_b8", "cityscapes_1024x2048_b8"):
        base = pkg.synthetic.make_workload_inputs(name, mode="model", seed=1, device=dev)
        inputs = {}
        for tag, dt in dtypes.items():
            d = dict(base)
            if dt != torch.float32:
                d["value"], d["grad_output"] = base["value"].to(dt), base["grad_output"].to(dt)
            else:   # the same values as the 16-bit arms see: rounded through bf16 once
                d["value"], d["grad_output"] = base["value"].bfloat16().float(), base["grad_output"].bfloat16().float()
            inputs[tag] = d
        del base

        def calls(tag):
            d = inputs[tag]
            a = (d["value"], d["spatial_shapes"], d["level_start_index"], d["sampling_locations"], d["attention_weights"])
            fwd = pkg.ms_deform_attn_forward if tag == "fp32" else pkg.ms_deform_attn_mixed_forward
            bwd = pkg.ms_deform_attn_backward if tag == "fp32" else pkg.ms_deform_attn_mixed_backward
            return {"forward": lambda: fwd(*a, 128),
                    "backward": lambda: bwd(*a, d["grad_output"], 128),
                    "fwd+bwd": lambda: (fwd(*a, 128), bwd(*a, d["grad_output"], 128))}

        arms = [(op, variant) for op, variant in (("forward", 0), ("backward", 0), ("backward", 20), ("backward", 2),
                                                  ("fwd+bwd", 0)) if op in ops]
        times = {(tag, op, v): [] for tag in dtypes for op, v in arms}
        fns = {tag: calls(tag) for tag in dtypes}
        for tag in dtypes:                                  # warm-up of every shape and arm
            for op, v in arms:
                pkg.set_option("bwd_variant", v)
                for _ in range(2):
                    fns[tag][op]()
        pkg.set_option("bwd_variant", 0)
        torch.cuda.synchronize()
        for _ in range(args.steps):
            for op, v in arms:
                pkg.set_option("bwd_variant", v)
                for tag in dtypes:                          # the types alternate
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    fns[tag][op]()
                    e1.record()
                    e1.synchronize()
                    times[(tag, op, v)].append(e0.elapsed_time(e1))
        pkg.set_option("bwd_variant", 0)
        for (tag, op, v), ts in times.items():
            b = op_bytes(inputs[tag], inputs[tag]["value"].element_size())
            nbytes = b["forward"] * (op != "backward") + b["backward"] * (op != "forward")
            ms = statistics.median(ts)
            emit({"part": "a", "label": args.label, "workload": name, "dtype": tag, "op": op,
                  "bwd_variant": {0: "gated default", 20: "merging forced", 2: "per-row forced"}[v],
                  "ms_median": ms, "ms_min": min(ts), "ms_max": max(ts), "timed_calls": len(ts),
                  "algorithmic_bytes": nbytes, "algorithmic_bytes_per_query": nbytes / b["queries"],
                  "accum_zero_fill_bytes": b["accum_zero_fill"] if op != "forward" else 0,
                  "accum_conversion_read_bytes": b["accum_conversion_read"] if op != "forward" else 0,
                  "algorithmic_GBs": nbytes / ms / 1e6, "l2": "evicted before every call (256 MB write)"})
        del inputs, fns
        torch.cuda.empty_cache()


def part_f(pkg, args, emit):
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    tags = [t for t in args.dtypes.split(",") if t != "fp32"]
    for name in ("cityscapes_512x1024_b8", "cityscapes_1024x2048_b8"):
        w = pkg.synthetic.WORKLOADS[name]
        levels, N, M, P = list(w.levels), w.batch, 8, 4
        L, S = len(levels), sum(h * wd for h, wd in levels)
        gen = torch.Generator(device=dev).manual_seed(1)
        base = {"value": torch.randn(N, S, M, 32, device=dev, generator=gen),
                "off": torch.randn(N, S, M, L, P, 2, device=dev, generator=gen) * 2.0,
                "logits": torch.randn(N, S, M, L * P, device=dev, generator=gen),
                "grad": torch.randn(N, S, M * 32, device=dev, generator=gen)}
        shapes, lsi = pkg.synthetic.level_tensors(levels, device=dev)
        ref = pkg.modules.reference_points_for(levels, dev)                 # [1, S, L, 2], fp32
        wh = shapes.flip(-1).float()[None, None, None, :, None, :]
        inputs = {"fp32": {k: v.bfloat16().float() for k, v in base.items()}}   # the values the 16-bit arms see
        for t in tags:
            inputs[t] = {k: v.to(DTYPES[t]) for k, v in base.items()}
        del base

        def fused(d):
            leaves = [d[k].requires_grad_(True) for k in ("value", "off", "logits")]
            return pkg.MSDeformAttnFusedFunction.apply(leaves[0], shapes, lsi, ref, leaves[1], leaves[2])

        def unfused(d):          # MSDeformAttn(fused=False) under autocast: fp32 producers, then the mixed op
            v, off, lg = (d[k].requires_grad_(True) for k in ("value", "off", "logits"))
            wts = torch.softmax(lg.float(), -1).view(N, S, M, L, P)
            loc = ref[:, :, None, :, None, :] + off.float() / wh
            return pkg.MSDeformAttnMixedFunction.apply(v, shapes, lsi, loc.contiguous(), wts.contiguous(), 128)

        arms = [("fp32", "fused", fused)] + [(t, kind, fn) for t in tags for kind, fn in (("fused", fused),
                                                                                         ("unfused", unfused))]
        times = {(t, k, op): [] for t, k, _ in arms for op in ("forward", "backward", "fwd+bwd")}

        def one(t, fn, op):
            d = inputs[t]
            if op == "forward":
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                with torch.no_grad():
                    e0.record()
                    fn(d)
                    e1.record()
            else:
                out = fn(d) if op == "backward" else None
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                if out is None:
                    out = fn(d)
                out.backward(d["grad"])
                e1.record()
                for k in ("value", "off", "logits"):
                    d[k].grad = None
            e1.synchronize()
            return e0.elapsed_time(e1)

        for t, _, fn in arms:                               # warm-up of every arm
            for op in ("forward", "backward", "fwd+bwd"):
                one(t, fn, op)
        for _ in range(args.steps):
            for op in ("forward", "backward", "fwd+bwd"):
                for t, k, fn in arms:                       # the arms alternate
                    times[(t, k, op)].append(one(t, fn, op))
        for (t, k, op), ts in times.items():
            emit({"part": "f", "label": args.label, "workload": name, "dtype": t, "producers": k, "op": op,
                  "ms_median": statistics.median(ts), "ms_min": min(ts), "ms_max": max(ts), "timed_calls": len(ts),
                  "what": "fused: MSDeformAttnFusedFunction on raw offsets / logits; unfused: torch fp32 softmax and "
                          "locations + MSDeformAttnMixedFunction (autograd, L*P = 12, offsets ~ N(0, 2) px)",
                  "l2": "evicted before every call (256 MB write)"})
        del inputs
        torch.cuda.empty_cache()


def _evicted(flush, fn):
    """Time one call of `fn` after a 256 MB write that evicts the L2 (events bracket the call only)."""
    flush.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def part_l(pkg, args, emit):
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    rows, cols = 344064, 256
    gen = torch.Generator(device=dev).manual_seed(4)
    x = torch.randn(rows, cols, device=dev, generator=gen)
    w = torch.rand(cols, device=dev, generator=gen) + 0.5
    b = torch.randn(cols, device=dev, generator=gen) * 0.1
    gy = torch.randn(rows, cols, device=dev, generator=gen)
    base_r = torch.randn(rows, cols, device=dev, generator=gen)
    base_g16 = torch.randn(rows, cols, device=dev, generator=gen)
    norm = torch.nn.LayerNorm(cols).to(dev)
    with torch.no_grad():
        norm.weight.copy_(w)
        norm.bias.copy_(b)
    for tag in ("bf16", "fp16"):
        dt = DTYPES[tag]
        r16, gy16 = base_r.to(dt), base_g16.to(dt)
        r32 = r16.float()

        def composition_fwd():
            with torch.no_grad(), torch.autocast("cuda", dtype=dt):
                y = norm(x + r16)
                y.to(dt)

        def composition_bwd():
            xl, rl = x.detach().requires_grad_(True), r16.detach().requires_grad_(True)
            with torch.autocast("cuda", dtype=dt):
                y = norm(xl + rl)
                y16 = y.to(dt)
            return lambda: torch.autograd.backward([y, y16], [gy, gy16])

        arms = {
            ("mixed kernels", "forward"): lambda: pkg.add_layernorm_mixed(x, r16, w, b),
            ("torch autocast composition", "forward"): composition_fwd,
            ("fp32 kernels", "forward"): lambda: pkg.add_layernorm(x, r32, w, b),
            ("mixed kernels", "backward"): lambda: pkg.ops.add_layernorm_mixed_backward(gy, gy16, x, r16, w),
            ("torch autocast composition", "backward"): None,
            ("fp32 kernels", "backward"): lambda: pkg.ops.add_layernorm_backward(gy, x, r32, w),
        }
        nbytes = {("mixed kernels", "forward"): 12, ("torch autocast composition", "forward"): 12,
                  ("fp32 kernels", "forward"): 12, ("mixed kernels", "backward"): 18,
                  ("torch autocast composition", "backward"): 18, ("fp32 kernels", "backward"): 16}
        times = {k: [] for k in arms}

        def one(k):
            if k == ("torch autocast composition", "backward"):
                bwd = composition_bwd()            # the forward runs untimed just before
                return _evicted(flush, bwd)
            return _evicted(flush, arms[k])
        for k in arms:
            for _ in range(2):
                one(k)
        for _ in range(args.steps):
            for k in arms:                                  # the arms alternate
                times[k].append(one(k))
        for (arm, op), ts in times.items():
            ms = statistics.median(ts)
            byt = nbytes[(arm, op)] * rows * cols
            emit({"part": "l", "what": "residual + LayerNorm site, 344064 x 256", "dtype": tag, "arm": arm, "op": op,
                  "ms_median": ms, "ms_min": min(ts), "ms_max": max(ts), "timed_calls": len(ts),
                  "algorithmic_bytes": byt, "algorithmic_GBs": byt / ms / 1e6,
                  "hbm_share": byt / ms / 1e6 / HBM_GBS, "hbm_GBs_reference": HBM_GBS,
                  "l2": "evicted before every call (256 MB write)"})


def part_p(pkg, args, emit):
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for name in ("cityscapes_512x1024_b8", "cityscapes_1024x2048_b8"):
        w = pkg.synthetic.WORKLOADS[name]
        levels, N, M, P = list(w.levels), w.batch, 8, 4
        L, S = len(levels), sum(h * wd for h, wd in levels)
        gen = torch.Generator(device=dev).manual_seed(1)
        value = torch.randn(N, S, M, 32, device=dev, generator=gen)
        proj = torch.cat((torch.randn(N, S, 2 * M * L * P, device=dev, generator=gen) * 2.0,
                          torch.randn(N, S, M * L * P, device=dev, generator=gen)), -1)
        table = torch.randn(S, 3 * M * L * P, device=dev, generator=gen) * 0.3
        shapes, lsi = pkg.synthetic.level_tensors(levels, device=dev)
        ref = pkg.modules.reference_points_for(levels, dev)
        arms = {}
        v32, p32 = value.bfloat16().float(), proj.bfloat16().float()
        arms["fp32 packed + table"] = lambda: pkg.ops.ms_deform_attn_fused_forward_packed(
            v32, shapes, lsi, ref, p32, L, P, query_table=table)
        for tag in ("bf16", "fp16"):
            dt = DTYPES[tag]
            v16, p16 = value.to(dt), proj.to(dt)
            off16 = p16[..., :2 * M * L * P].reshape(N, S, M, L, P, 2).contiguous()
            lg16 = p16[..., 2 * M * L * P:].reshape(N, S, M, L * P).contiguous()
            arms[f"{tag} packed + table"] = (lambda v16=v16, p16=p16: pkg.ops.ms_deform_attn_fused_mixed_forward_packed(
                v16, shapes, lsi, ref, p16, L, P, query_table=table))
            arms[f"{tag} fused, separate tensors"] = (lambda v16=v16, o=off16, g=lg16: pkg.ms_deform_attn_fused_forward(
                v16, shapes, lsi, ref, o, g))
        times = {k: [] for k in arms}
        for k, fn in arms.items():
            for _ in range(2):
                fn()
        for _ in range(args.steps):
            for k, fn in arms.items():                      # the arms alternate
                times[k].append(_evicted(flush, fn))
        for k, ts in times.items():
            emit({"part": "p", "workload": name, "arm": k, "ms_median": statistics.median(ts), "ms_min": min(ts),
                  "ms_max": max(ts), "timed_calls": len(ts), "l2": "evicted before every call (256 MB write)"})
        del arms, value, proj, v32, p32
        torch.cuda.empty_cache()


def part_g(pkg, args, emit):
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    N, C, G, eps = 8, 256, 32, 1e-5
    gen = torch.Generator(device=dev).manual_seed(6)
    w = torch.rand(C, device=dev, generator=gen) + 0.5
    b = torch.randn(C, device=dev, generator=gen) * 0.1
    cb = torch.randn(C, device=dev, generator=gen) * 0.1
    base = torch.randn(N, C, 256, 512, device=dev, generator=gen) * 2 + 0.5
    up = torch.randn(N, C, 128, 256, device=dev, generator=gen)
    cot = torch.randn(N, C, 256, 512, device=dev, generator=gen)
    levels = [(128, 256), (64, 128), (32, 64)]
    S = sum(h * wd for h, wd in levels)
    proj = [torch.randn(N, C, h, wd, device=dev, generator=gen) for h, wd in levels]
    rows_cot = torch.randn(N, S, C, device=dev, generator=gen)
    norm = torch.nn.GroupNorm(G, C, eps=eps).to(dev)
    with torch.no_grad():
        norm.weight.copy_(w)
        norm.bias.copy_(b)
    for tag in ("bf16", "fp16"):
        dt = DTYPES[tag]
        x16, g16 = base.to(dt), cot.to(dt)
        x32, g32 = x16.float(), g16.float()
        p16 = [p.to(dt) for p in proj]
        p32 = [p.float() for p in p16]
        rows = torch.empty(N, S, C, device=dev)
        starts = [0]
        for h, wd in levels:
            starts.append(starts[-1] + h * wd)
        slices = [rows[:, a:z] for a, z in zip(starts, starts[1:])]
        gslices = [rows_cot[:, a:z] for a, z in zip(starts, starts[1:])]
        sites = {}
        for site, relu, u in (("lateral", False, up), ("output", True, None)):
            _, st16 = pkg.ops.group_norm_train(x16, w, b, G, eps, relu=relu, up=u)
            ups = tuple(u.shape[-2:]) if u is not None else None

            def comp(relu=relu, u=u):
                xl = x16.detach().requires_grad_(True)
                ul = u.detach().requires_grad_(True) if u is not None else None
                wl, bl = w.detach().requires_grad_(True), b.detach().requires_grad_(True)
                with torch.autocast("cuda", dtype=dt):
                    y = F.group_norm(xl, G, wl, bl, eps)
                    y = torch.relu(y) if relu else y
                    if ul is not None:
                        y = y + F.interpolate(ul, size=xl.shape[-2:], mode="bilinear", align_corners=False)
                    y = y.to(dt)
                return y
            sites[site] = {
                ("16-bit kernels", "forward"): lambda relu=relu, u=u: pkg.ops.group_norm_train(
                    x16, w, b, G, eps, relu=relu, up=u, out_dtype=dt),
                ("torch autocast composition", "forward"): lambda comp=comp: comp(),
                ("fp32 kernels", "forward"): lambda relu=relu, u=u: pkg.ops.group_norm_train(x32, w, b, G, eps,
                                                                                            relu=relu, up=u),
                ("16-bit kernels", "backward"): lambda relu=relu, st=st16, ups=ups: pkg.ops.group_norm_backward(
                    g16, x16, w, b, st, G, relu=relu, up_shape=ups),
                ("torch autocast composition", "backward"): ("graph", lambda comp=comp: comp(), g16),
                ("fp32 kernels", "backward"): lambda relu=relu, st=st16, ups=ups: pkg.ops.group_norm_backward(
                    g32, x32, w, b, st, G, relu=relu, up_shape=ups),
            }
        stats16 = [pkg.ops.group_norm_rows_train(p, w, b, G, eps, r, channel_bias=cb) for p, r in zip(p16, slices)]

        def rows_comp():
            leaves = [p.detach().requires_grad_(True) for p in p16]
            wl, bl = w.detach().requires_grad_(True), b.detach().requires_grad_(True)
            with torch.autocast("cuda", dtype=dt):
                return torch.cat([F.group_norm(p, G, wl, bl, eps).flatten(2).transpose(1, 2) for p in leaves], 1)
        sites["input projections"] = {
            ("16-bit kernels", "forward"): lambda: [pkg.ops.group_norm_rows_train(p, w, b, G, eps, r, channel_bias=cb)
                                                    for p, r in zip(p16, slices)],
            ("torch autocast composition", "forward"): rows_comp,
            ("fp32 kernels", "forward"): lambda: [pkg.ops.group_norm_rows_train(p, w, b, G, eps, r, channel_bias=cb)
                                                  for p, r in zip(p32, slices)],
            ("16-bit kernels", "backward"): lambda: [pkg.ops.group_norm_rows_backward(
                g, p, w, b, st, G, channel_bias=cb, with_channel_bias=True) for g, p, st in zip(gslices, p16, stats16)],
            ("torch autocast composition", "backward"): ("graph", rows_comp, rows_cot),
            ("fp32 kernels", "backward"): lambda: [pkg.ops.group_norm_rows_backward(
                g, p, w, b, st, G, channel_bias=cb, with_channel_bias=True) for g, p, st in zip(gslices, p32, stats16)],
        }
        elems = {"lateral": x16.numel(), "output": x16.numel(), "input projections": N * S * C}
        upel = up.numel()
        # bytes of the 16-bit kernels and of the fp32 kernels per site and op (see the docstring)
        nbytes = {("lateral", "forward"): (6 * elems["lateral"] + 4 * upel, 12 * elems["lateral"] + 4 * upel),
                  ("output", "forward"): (6 * elems["output"], 12 * elems["output"]),
                  ("input projections", "forward"): (8 * elems["input projections"], 12 * elems["input projections"]),
                  ("lateral", "backward"): (10 * elems["lateral"] + 6 * upel, 20 * elems["lateral"] + 8 * upel),
                  ("output", "backward"): (10 * elems["output"], 20 * elems["output"]),
                  ("input projections", "backward"): (16 * elems["input projections"],
                                                      20 * elems["input projections"])}
        for site, arms in sites.items():
            def one(k, arms=arms):
                fn = arms[k]
                if isinstance(fn, tuple):                      # autograd: the forward untimed, then the backward
                    y = fn[1]()
                    return _evicted(flush, lambda: y.backward(fn[2]))
                return _evicted(flush, fn)
            times = {k: [] for k in arms}
            for k in arms:
                for _ in range(2):
                    one(k)
            for _ in range(args.steps):
                for k in arms:                              # the arms alternate
                    times[k].append(one(k))
            for (arm, op), ts in times.items():
                ms = statistics.median(ts)
                byt = nbytes[(site, op)][1 if arm == "fp32 kernels" else 0]
                emit({"part": "g", "what": f"GroupNorm site '{site}', 1024x2048 batch 8, Swin-T, conv_dim 256",
                      "dtype": tag, "arm": arm, "op": op, "ms_median": ms, "ms_min": min(ts), "ms_max": max(ts),
                      "timed_calls": len(ts), "algorithmic_bytes": byt,
                      "bytes_per_element": byt / elems[site], "algorithmic_GBs": byt / ms / 1e6,
                      "hbm_share": byt / ms / 1e6 / HBM_GBS, "hbm_GBs_reference": HBM_GBS,
                      "l2": "evicted before every call (256 MB write)"})
        del sites, x16, g16, x32, g32, p16, p32, rows
        torch.cuda.empty_cache()


@contextlib.contextmanager
def gn16_off(pkg):
    """The 16-bit GroupNorm kernels off: the predicates refuse bf16 / fp16 maps, so the decoder's linear="autocast"
    path runs torch's GroupNorms as before those kernels."""
    names = ("group_norm_supported", "group_norm_rows_supported", "channel_bias_supported")
    saved = {n: getattr(pkg.ops, n) for n in names}
    for n, f in saved.items():
        setattr(pkg.ops, n, lambda x, *a, _f=f, **k: x.dtype == torch.float32 and _f(x, *a, **k))
    try:
        yield
    finally:
        for n, f in saved.items():
            setattr(pkg.ops, n, f)


OFF = ", 16-bit GroupNorm kernels off"
LIN_OFF = ", 16-bit Linear kernels off"


@contextlib.contextmanager
def linear16_off(pkg):
    """The 16-bit Linear kernels off: their predicates refuse every shape, so linear="autocast" runs torch's autocast
    GEMMs (and the FFN's separate ReLU) as before those kernels."""
    fn, op = pkg.functions.LinearMixedFunction, pkg.ops.linear_mixed_supported
    saved = fn.__dict__["supported"]
    fn.supported = staticmethod(lambda *a, **k: False)
    pkg.ops.linear_mixed_supported = lambda *a, **k: False
    try:
        yield
    finally:
        fn.supported = saved
        pkg.ops.linear_mixed_supported = op


def _switch(pkg, tag):
    return gn16_off(pkg) if tag.endswith(OFF) else linear16_off(pkg) if tag.endswith(LIN_OFF) \
        else contextlib.nullcontext()


def _decoder(pkg, fused, linear, amp, train):
    torch.manual_seed(0)
    m = pkg.pixel_decoder.MSDeformAttnPixelDecoder(
        SWIN_T, transformer_dropout=0.1 if train else 0.0, transformer_nheads=8, transformer_dim_feedforward=1024,
        transformer_enc_layers=6, conv_dim=256, mask_dim=256, norm="GN", transformer_in_features=["res3", "res4", "res5"],
        common_stride=4, fused=fused, linear=linear, amp=amp).cuda()
    return m.train() if train else m.eval()


def _feats(batch, h, w, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return {k: torch.randn(batch, c, h // s, w // s, device="cuda", generator=gen) for k, (c, s) in SWIN_T.items()}


def part_b(pkg, args, emit):
    feats = _feats(8, 1024, 2048, 3)
    arms = [("fp32 fused tf32x3", dict(fused=True, linear="tf32x3", amp=False), None),
            ("amp bf16", dict(fused=True, linear="torch", amp=True), torch.bfloat16),
            ("amp bf16 fused=False", dict(fused=False, linear="torch", amp=True), torch.bfloat16),
            ("amp bf16 linear=autocast", dict(fused=True, linear="autocast", amp=True), torch.bfloat16),
            ("amp bf16 linear=autocast" + OFF, dict(fused=True, linear="autocast", amp=True), torch.bfloat16),
            ("amp bf16 linear=autocast" + LIN_OFF, dict(fused=True, linear="autocast", amp=True), torch.bfloat16)]
    models = {tag: _decoder(pkg, train=False, **kw) for tag, kw, _ in arms}
    res = {tag: [] for tag, _, _ in arms}
    for _ in range(args.repeats):
        for tag, _, dt in arms:
            ctx = torch.autocast("cuda", dtype=dt) if dt is not None else contextlib.nullcontext()

            def fwd(m=models[tag], ctx=ctx, tag=tag):
                with torch.no_grad(), ctx, _switch(pkg, tag):
                    m.forward_features(feats)
            res[tag].append(timed(fwd, max(2, args.steps // 4), 2))
    for tag, _, _ in arms:
        emit({"part": "b", "what": "pixel-decoder forward_features, no autograd, 1024x2048, batch 8, Swin-T pyramid, "
                                   "6 encoder layers", "arm": tag, "ms": min(res[tag]), "ms_all_repeats": res[tag]})


def part_c(pkg, args, emit):
    feats = _feats(16, 512, 1024, 2)
    arms = [("fp32 fused tf32x3", dict(fused=True, linear="tf32x3", amp=False), None),
            ("amp bf16", dict(fused=True, linear="torch", amp=True), torch.bfloat16),
            ("amp bf16 fused=False", dict(fused=False, linear="torch", amp=True), torch.bfloat16),
            ("amp bf16 linear=autocast", dict(fused=True, linear="autocast", amp=True), torch.bfloat16),
            ("amp bf16 linear=autocast" + OFF, dict(fused=True, linear="autocast", amp=True), torch.bfloat16),
            ("amp bf16 linear=autocast" + LIN_OFF, dict(fused=True, linear="autocast", amp=True), torch.bfloat16),
            ("amp fp16 + GradScaler", dict(fused=True, linear="torch", amp=True), torch.float16),
            ("amp fp16 + GradScaler fused=False", dict(fused=False, linear="torch", amp=True), torch.float16),
            ("amp fp16 + GradScaler linear=autocast", dict(fused=True, linear="autocast", amp=True), torch.float16),
            ("amp fp16 + GradScaler linear=autocast" + OFF, dict(fused=True, linear="autocast", amp=True),
             torch.float16),
            ("amp fp16 + GradScaler linear=autocast" + LIN_OFF, dict(fused=True, linear="autocast", amp=True),
             torch.float16)]
    steps = {}
    for tag, kw, dt in arms:
        m = _decoder(pkg, train=True, **kw)
        opt = torch.optim.AdamW(m.parameters(), lr=1e-4)
        scaler = torch.amp.GradScaler("cuda") if dt == torch.float16 else None
        ctx = (lambda dt=dt: torch.autocast("cuda", dtype=dt)) if dt is not None else contextlib.nullcontext

        def step(m=m, opt=opt, scaler=scaler, ctx=ctx, tag=tag):
            opt.zero_grad(set_to_none=True)
            with ctx(), _switch(pkg, tag):
                mask, low, multi = m.forward_features(feats)
                loss = sum(o.float().square().mean() for o in (mask, low, *multi))
            if scaler is None:
                loss.backward()
                opt.step()
            else:
                scaler.scale(loss).backward()
                scaler.step(opt)
                scaler.update()
        steps[tag] = step
    res, peak = {tag: [] for tag, _, _ in arms}, {}
    for r in range(args.repeats):
        for tag, _, _ in arms:                               # the arms alternate
            torch.cuda.reset_peak_memory_stats()
            res[tag].append(timed(steps[tag], max(2, args.steps // 4), args.warmup if r == 0 else 1))
            peak[tag] = max(peak.get(tag, 0.0), torch.cuda.max_memory_allocated() / 2 ** 30)
    for tag, _, _ in arms:
        ms = min(res[tag])
        emit({"part": "c", "what": "pixel-decoder training step (forward_features + loss + backward + AdamW), "
                                   "512x1024, batch 16, Swin-T pyramid, 6 encoder layers", "arm": tag, "ms": ms,
              "ms_all_repeats": res[tag], "images_per_s": 16 / ms * 1e3, "peak_mem_gib": peak[tag],
              "note": "peak memory includes the parameters and optimizer state of all arms' models"})


# the encoder's Linear sites (d = 256, 8 heads, 4 levels x 4 points, FFN 1024): (name, in, out, relu)
LINEAR_SITES = [("value / output projection", 256, 256, False), ("query GEMM (offsets + logits)", 256, 288, False),
                ("sampling offsets", 256, 192, False), ("attention weights", 256, 96, False),
                ("linear1 + ReLU", 256, 1024, True), ("linear2", 1024, 256, False)]


def part_m(pkg, args, emit):
    """The 16-bit Linear kernels against torch's autocast composition at the encoder's Linear sites: forward, input
    gradient, weight + bias gradient; median of `--steps` alternating calls, the L2 evicted before each."""
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for rows in (344064, 172032):
        for tag in ("bf16", "fp16"):
            dt = DTYPES[tag]
            for name, k, n, relu in LINEAR_SITES:
                gen = torch.Generator(device=dev).manual_seed(k + n)
                x16 = torch.randn(rows, k, device=dev, generator=gen).to(dt)
                g16 = (torch.randn(rows, n, device=dev, generator=gen) * 1e-2).to(dt)
                w = torch.randn(n, k, device=dev, generator=gen) / k ** 0.5
                b = torch.randn(n, device=dev, generator=gen) * 0.1
                w16, wt16 = w.to(dt), w.t().contiguous().to(dt)

                def torch_fwd():
                    with torch.no_grad(), torch.autocast("cuda", dtype=dt):
                        y = F.linear(x16, w, b)
                        return F.relu(y) if relu else y

                def addmm_act():
                    with torch.no_grad(), torch.autocast("cuda", dtype=dt):
                        return torch._addmm_activation(b.to(dt), x16, w16.t())

                def torch_wgrad():
                    return (g16.t() @ x16).float(), g16.sum(0).float()

                arms = {("16-bit kernels", "forward"): lambda: pkg.ops.linear_mixed(x16, w16, b, relu=relu),
                        ("torch autocast composition", "forward"): torch_fwd,
                        ("16-bit kernels", "input gradient"): lambda: pkg.ops.linear_mixed(g16, wt16),
                        ("torch autocast composition", "input gradient"): lambda: g16 @ w16,
                        ("16-bit kernels", "weight + bias gradient"): lambda: pkg.ops.linear_mixed_wgrad(g16, x16),
                        ("torch autocast composition", "weight + bias gradient"): torch_wgrad}
                if relu:
                    try:
                        addmm_act()
                        arms[("torch._addmm_activation (cuBLASLt ReLU epilogue)", "forward")] = addmm_act
                    except RuntimeError as e:
                        emit({"part": "m", "site": name, "dtype": tag, "note": f"_addmm_activation: {e}"[:300]})
                act = rows * (k + n) * 2
                nbytes = {"forward": act + n * k * 2, "input gradient": act + n * k * 2,
                          "weight + bias gradient": act + n * k * 4 + n * 4}
                times = {a: [] for a in arms}
                for a in arms:
                    for _ in range(2):
                        _evicted(flush, arms[a])
                for _ in range(args.steps):
                    for a in arms:                                  # the arms alternate
                        times[a].append(_evicted(flush, arms[a]))
                for (arm, op), ts in times.items():
                    ms = statistics.median(ts)
                    emit({"part": "m", "site": name, "rows": rows, "in": k, "out": n, "relu": relu, "dtype": tag,
                          "arm": arm, "op": op, "ms_median": ms, "ms_min": min(ts), "ms_max": max(ts),
                          "timed_calls": len(ts), "algorithmic_bytes": nbytes[op],
                          "algorithmic_GBs": nbytes[op] / ms / 1e6, "hbm_share": nbytes[op] / ms / 1e6 / HBM_GBS,
                          "hbm_GBs_reference": HBM_GBS, "l2": "evicted before every call (256 MB write)"})
                del x16, g16
                torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="a,b,c", help="a, b, c: profiles/r5_mixed.jsonl; f, b, c: r6_fused_mixed.jsonl; "
                                                  "l, p, b, c: r7_autocast_encoder.jsonl; g, b, c: r8_group_norm_mixed.jsonl; "
                                                  "m, b, c: r9_linear_mixed.jsonl")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dtypes", default="fp32,bf16,fp16", help="part (a): element types of value")
    ap.add_argument("--ops", default="forward,backward,fwd+bwd", help="part (a): calls timed")
    ap.add_argument("--label", default="", help="part (a): recorded in every line (e.g. the library build)")
    ap.add_argument("--repeats", type=int, default=3, help="parts (b), (c): alternating repeats of each arm (min reported)")
    ap.add_argument("--out", default=os.path.join(os.environ.get("BENCH_OUT") or os.path.join(ROOT, "bench_out"),
                                                  "mixed"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_mixed.py measures on a CUDA device; none is available")
    pkg = load_package()
    os.makedirs(args.out, exist_ok=True)
    info = card()
    path = os.path.join(args.out, "mixed.jsonl")

    def emit(rec):
        rec = {**info, **rec}
        print(json.dumps(rec), flush=True)
        with open(path, "a") as f:
            f.write(json.dumps(rec) + "\n")
    for part in args.parts.split(","):
        {"a": part_a, "f": part_f, "b": part_b, "c": part_c, "l": part_l, "p": part_p, "g": part_g, "m": part_m}[part](pkg, args, emit)


if __name__ == "__main__":
    main()
