"""Cost of the deterministic mode (torch.use_deterministic_algorithms(True)) on the B200: every measurement runs
the same work with the flag off and on, alternating in one process.

    python tools/bench_deterministic.py [--parts msda,linear,steps] [--steps 10] [--out DIR]

DIR defaults to $BENCH_OUT/deterministic, and BENCH_OUT to bench_out/ in the repository (git-ignored).

msda    the MSDA backward at configs[1] (512x1024 pyramid, batch 8, model-like locations), plain
        (ms_deform_attn_backward) and fused (ms_deform_attn_fused_backward), with the L2 evicted before every
        call (a 256 MB buffer is overwritten: the inputs then come from HBM, as inside a training step).  For the
        deterministic arm a separate torch.profiler run splits the call into its stages: records kernel, sort (all
        CUB kernels), bucket bounds, gather, and torch's fill of the freshly allocated workspace and outputs
        (torch.utils.deterministic.fill_uninitialized_memory).
linear  linear_wgrad at 172 032 x 256 x 256 and the residual + LayerNorm backward at 344 064 x 256, L2 evicted.
steps   the encoder training step of configs[4] (512x1024, batch 16, 6 layers, fused producers, linear="tf32x3",
        dropout 0.1, AdamW) and the pixel-decoder training step at 512x1024, batch 16 (as tools/bench_decoder_train.py
        part b, shipped arm).

Timing: CUDA events; the minimum over --repeats alternating repeats is reported with all repeats.  Every JSON line
carries the card's name and power limit, read in the same run (read-only `nvidia-smi --query-gpu`).
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from __graft_entry__ import load_package  # noqa: E402
from bench_decoder_train import card  # noqa: E402

STAGES = (("records", ("msda_bwd_d32_kernel", "msda_bwd_generic_kernel")),
          ("sort", ("DeviceRadixSort", "Onesweep", "cub::")),
          ("bounds", ("msda_det_bounds",)),
          ("gather", ("msda_det_gather",)),
          ("fill", ("fill", "Fill")))


def set_flag(on):
    torch.use_deterministic_algorithms(on)


def timed(fn, steps, warm, flush=None):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    total = 0.0
    for _ in range(steps):
        if flush is not None:
            flush.zero_()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1)
    return total / steps


def alternate(fn, args, flush=None):
    res = {False: [], True: []}
    for _ in range(args.repeats):
        for on in (False, True):
            set_flag(on)
            res[on].append(timed(fn, args.steps, args.warmup, flush))
    set_flag(False)
    return {"off": res[False], "on": res[True]}


def stages(fn, calls=5):
    """Device time per stage of one deterministic call (torch.profiler, a run of its own)."""
    set_flag(True)
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    set_flag(False)
    out = {name: 0.0 for name, _ in STAGES}
    out["other"] = 0.0
    for evt in prof.key_averages():
        us = getattr(evt, "device_time_total", None)
        if us is None:
            us = evt.cuda_time_total
        stage = next((name for name, keys in STAGES if any(k in evt.key for k in keys)), "other")
        out[stage] += us / calls / 1e3
    return {k: round(v, 4) for k, v in out.items()}


def summary(rec, res):
    rec["ms_off"], rec["ms_on"] = min(res["off"]), min(res["on"])
    rec["on_over_off"] = rec["ms_on"] / rec["ms_off"]
    rec["ms_all_repeats"] = res
    return rec


def part_msda(pkg, args, emit, flush):
    dev = torch.device("cuda", 0)
    syn = pkg.synthetic
    d = syn.make_workload_inputs("cityscapes_512x1024_b8", mode="model", seed=1, device=dev)
    a = (d["value"], d["spatial_shapes"], d["level_start_index"], d["sampling_locations"], d["attention_weights"])
    N, Lq, M, L, P, _ = d["sampling_locations"].shape
    records = N * Lq * M * L * P * 4
    plain = lambda: pkg.ms_deform_attn_backward(*a, d["grad_output"], 128)          # noqa: E731
    levels = syn.WORKLOADS["cityscapes_512x1024_b8"].levels
    gen = torch.Generator(device=dev).manual_seed(2)
    ref = pkg.modules.reference_points_for(levels, dev).contiguous()
    off = torch.randn(N, Lq, M, L, P, 2, device=dev, generator=gen) * 2.0
    logits = torch.randn(N, Lq, M, L * P, device=dev, generator=gen)
    fused = lambda: pkg.ms_deform_attn_fused_backward(d["value"], d["spatial_shapes"], d["level_start_index"],  # noqa: E731
                                                      ref, off, logits, d["grad_output"])
    ws = pkg._lib.lib.msda_b200_backward_deterministic_workspace_bytes(N, d["value"].size(1), M, 32, L, Lq, P, 4)
    for kind, fn in (("plain", plain), ("fused", fused)):
        res = alternate(fn, args, flush)
        emit(summary({"part": "msda", "what": f"MSDA {kind} backward, configs[1] (512x1024 pyramid, batch 8), L2 evicted",
                      "records": records, "workspace_bytes": ws, "stages_ms_on": stages(fn)}, res))


def part_linear(pkg, args, emit, flush):
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(3)
    gy = torch.randn(172032, 256, device=dev, generator=gen)
    x = torch.randn(172032, 256, device=dev, generator=gen)
    emit(summary({"part": "linear", "what": "linear_wgrad 172032 x 256 x 256 (grad_W and grad_b), L2 evicted"},
                 alternate(lambda: pkg.ops.linear_wgrad(gy, x), args, flush)))
    del gy, x
    gy, x, r = (torch.randn(344064, 256, device=dev, generator=gen) for _ in range(3))
    w = torch.randn(256, device=dev, generator=gen) + 1
    emit(summary({"part": "linear", "what": "add_layernorm backward 344064 x 256, L2 evicted"},
                 alternate(lambda: pkg.ops.add_layernorm_backward(gy, x, r, w, 1e-5), args, flush)))


def part_steps(pkg, args, emit):
    dev = torch.device("cuda", 0)
    syn = pkg.synthetic
    levels, batch = syn.pyramid(512, 1024), 16
    torch.manual_seed(0)
    m = pkg.modules.MSDeformAttnTransformerEncoderOnly(
        d_model=256, nhead=8, num_encoder_layers=6, dim_feedforward=1024, dropout=0.1, num_feature_levels=3,
        enc_n_points=4, fused=True, linear="tf32x3").to(dev).train()
    with torch.no_grad():
        for layer in m.encoder.layers:
            torch.nn.init.normal_(layer.self_attn.sampling_offsets.weight, std=0.02)
            torch.nn.init.normal_(layer.self_attn.attention_weights.weight, std=0.05)
    gen = torch.Generator(device=dev).manual_seed(20)
    srcs = [torch.randn(batch, 256, h, w, device=dev, generator=gen) for h, w in levels]
    pos = [torch.randn(batch, 256, h, w, device=dev, generator=gen) * 0.1 for h, w in levels]
    opt = torch.optim.AdamW(m.parameters(), lr=1e-4)

    def enc_step():
        opt.zero_grad(set_to_none=True)
        m(srcs, pos)[0].square().mean().backward()
        opt.step()
    emit(summary({"part": "steps", "what": "encoder training step (fwd+bwd+AdamW), configs[4]: 512x1024, batch 16, "
                                           "6 layers, fused producers, linear=tf32x3, dropout 0.1"},
                 alternate(enc_step, args)))
    del m, opt, srcs, pos
    torch.cuda.empty_cache()
    shapes = {"res2": (96, 4), "res3": (192, 8), "res4": (384, 16), "res5": (768, 32)}
    feats = {k: torch.randn(batch, c, 512 // s, 1024 // s, device=dev, generator=gen) for k, (c, s) in shapes.items()}
    torch.manual_seed(0)
    dec = pkg.pixel_decoder.MSDeformAttnPixelDecoder(
        shapes, transformer_dropout=0.1, transformer_nheads=8, transformer_dim_feedforward=1024,
        transformer_enc_layers=6, conv_dim=256, mask_dim=256, norm="GN", transformer_in_features=["res3", "res4", "res5"],
        common_stride=4, fused=True, linear="tf32x3").to(dev).train()
    opt = torch.optim.AdamW(dec.parameters(), lr=1e-4)

    def dec_step():
        opt.zero_grad(set_to_none=True)
        mask, low, multi = dec.forward_features(feats)
        sum(o.square().mean() for o in (mask, low, *multi)).backward()
        opt.step()
    cudnn = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True        # both arms: the flag itself does not change the convolutions
    try:
        emit(summary({"part": "steps", "what": "pixel-decoder training step (forward_features + loss + backward + AdamW), "
                                               "512x1024, batch 16, Swin-T pyramid, 6 encoder layers, linear=tf32x3, "
                                               "cudnn.deterministic"},
                     alternate(dec_step, args)))
    finally:
        torch.backends.cudnn.deterministic = cudnn


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="msda,linear,steps")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(os.environ.get("BENCH_OUT") or os.path.join(ROOT, "bench_out"),
                                                  "deterministic"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_deterministic.py measures on a CUDA device; none is available")
    os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    pkg = load_package()
    info = card()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "deterministic.jsonl")

    def emit(rec):
        rec.update(info)
        with open(path, "a") as f:
            f.write(json.dumps(rec) + "\n")
        print(json.dumps(rec), flush=True)
    flush = torch.empty(64 * 2 ** 20, dtype=torch.float32, device="cuda:0")      # 256 MB > 126 MB of L2
    parts = args.parts.split(",")
    if "msda" in parts:
        part_msda(pkg, args, emit, flush)
    if "linear" in parts:
        part_linear(pkg, args, emit, flush)
    if "steps" in parts:
        part_steps(pkg, args, emit)


if __name__ == "__main__":
    main()
