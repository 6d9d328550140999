"""Training cost of the pixel decoder's GroupNorms on the B200: the fused kernels (GroupNormFunction /
GroupNormRowsFunction) against torch eager autograd.

    python tools/bench_decoder_train.py [--parts a,b] [--steps 10] [--out DIR]

DIR defaults to $BENCH_OUT/decoder_train, and BENCH_OUT to bench_out/ in the repository (git-ignored).

(a) kernel level: training forward + backward of one stride-4 map of the 512x1024 / batch 16 training shape
    (x = 16 x 256 x 128 x 256 fp32, 134 M elements), as the FPN lateral (GroupNorm + bilinear up-sampled add of a
    16 x 256 x 64 x 128 map, gradients of x, gamma, beta and the up-sampled map) and as the output convolution's
    epilogue (GroupNorm + ReLU), each against torch eager autograd of the same expression.  Algorithmic bytes per
    element (x, grad_y, y, grad_x once each where they must move; the up-sampled map is 1/4 of the elements):
        fused  lateral 12 + 1 forward, 20 + 5 backward = 38;  output 12 forward, 20 backward = 32
        torch  lateral 52, output 52 (the counts of DESIGN.md section 10)
    The maps (537 MB each) are far larger than the 126 MB L2: every pass reads HBM.
(b) whole step: MSDeformAttnPixelDecoder forward_features -> loss on all outputs -> backward -> AdamW at 512x1024,
    batch 16, Swin-T pyramid (as tools/bench_configs.py), for linear="torch", linear="tf32x3" with the GroupNorm
    kernels forced off, and linear="tf32x3" as shipped.

Timing: CUDA events around warmed repeats.  Every JSON line carries the card's name and power limit (read-only
`nvidia-smi --query-gpu=name,power.limit`) and the HBM peak it divides by.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from __graft_entry__ import load_package  # noqa: E402
from bench import measured_peak  # noqa: E402

BYTES = {("fused", "lateral"): 38, ("fused", "output"): 32, ("torch", "lateral"): 52, ("torch", "output"): 52}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:          # the numbers stay valid; say that the card was not identified
        return {"gpu": f"unknown ({e})", "power_limit": "unknown"}


def timed(fn, steps, warm):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def part_a(pkg, args, emit, peak):
    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(1)
    N, C, H, W, G = 16, 256, 128, 256, 32
    x = (torch.randn(N, C, H, W, device=dev, generator=gen) * 2 + 1).requires_grad_(True)
    cot = torch.randn(N, C, H, W, device=dev, generator=gen)
    w = (torch.randn(C, device=dev, generator=gen) * 0.3 + 1).requires_grad_(True)
    b = (torch.randn(C, device=dev, generator=gen) * 0.5).requires_grad_(True)
    up = torch.randn(N, C, H // 2, W // 2, device=dev, generator=gen).requires_grad_(True)
    for role in ("lateral", "output"):
        u, relu = (up, False) if role == "lateral" else (None, True)

        def fused():
            y = pkg.GroupNormFunction.apply(x, w, b, None, u, G, 1e-5, relu)
            y.backward(cot)

        def eager():
            y = F.group_norm(x, G, w, b, 1e-5)
            y = torch.relu(y) if relu else y
            if u is not None:
                y = y + F.interpolate(u, size=(H, W), mode="bilinear", align_corners=False)
            y.backward(cot)
        # alternate the two arms, so that other work on the host affects both alike
        res = {"fused": [], "torch": []}
        for _ in range(args.repeats):
            for name, fn in (("fused", fused), ("torch", eager)):
                res[name].append(timed(fn, args.steps, args.warmup))
        for name in ("fused", "torch"):
            ms = min(res[name])
            gbs = N * C * H * W * BYTES[(name, role)] / ms / 1e6
            emit({"part": "a", "map": role, "impl": name, "shape": [N, C, H, W],
                  "up_shape": list(up.shape) if u is not None else None, "relu": relu,
                  "ms_fwd_bwd": ms, "ms_all_repeats": res[name], "algorithmic_bytes_per_element": BYTES[(name, role)],
                  "algorithmic_GBs": gbs, "frac_of_hbm_peak": gbs / peak})
        x.grad = w.grad = b.grad = up.grad = None


def part_b(pkg, args, emit):
    dev = torch.device("cuda", 0)
    shapes = {"res2": (96, 4), "res3": (192, 8), "res4": (384, 16), "res5": (768, 32)}     # Swin-T
    gen = torch.Generator(device=dev).manual_seed(2)
    batch, (Himg, Wimg) = 16, (512, 1024)
    feats = {k: torch.randn(batch, c, Himg // s, Wimg // s, device=dev, generator=gen) for k, (c, s) in shapes.items()}
    arms = [("torch", False, False), ("tf32x3", True, False), ("tf32x3", True, True)]
    for linear, fused, gn_kernels in arms:
        torch.manual_seed(0)
        m = pkg.pixel_decoder.MSDeformAttnPixelDecoder(
            shapes, transformer_dropout=0.1, transformer_nheads=8, transformer_dim_feedforward=1024,
            transformer_enc_layers=6, conv_dim=256, mask_dim=256, norm="GN",
            transformer_in_features=["res3", "res4", "res5"], common_stride=4, fused=fused, linear=linear).to(dev).train()
        opt = torch.optim.AdamW(m.parameters(), lr=1e-4)
        saved = pkg.ops.group_norm_supported, pkg.ops.group_norm_rows_supported
        if not gn_kernels:
            pkg.ops.group_norm_supported = pkg.ops.group_norm_rows_supported = lambda *a, **k: False
        try:
            def step():
                opt.zero_grad(set_to_none=True)
                mask, low, multi = m.forward_features(feats)
                sum(o.square().mean() for o in (mask, low, *multi)).backward()
                opt.step()
            n0 = pkg.launch_count()
            step()
            launches = pkg.launch_count() - n0
            ms = timed(step, args.steps, args.warmup)
            peak_mem = torch.cuda.max_memory_allocated(dev) / 2 ** 30
        finally:
            pkg.ops.group_norm_supported, pkg.ops.group_norm_rows_supported = saved
        emit({"part": "b", "what": "pixel-decoder training step (forward_features + loss + backward + AdamW), "
                                   "512x1024, batch 16, Swin-T pyramid, 6 encoder layers",
              "linear": linear, "fused_producers": fused, "group_norm_kernels": gn_kernels, "ms": ms,
              "images_per_s": batch / ms * 1e3, "library_launches_per_step": launches, "peak_mem_gib": peak_mem})
        del m, opt
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parts", default="a,b")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=3, help="part (a): alternating repeats of each arm (min reported)")
    ap.add_argument("--out", default=os.path.join(os.environ.get("BENCH_OUT") or os.path.join(ROOT, "bench_out"),
                                                  "decoder_train"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_decoder_train.py measures on a CUDA device; none is available")
    pkg = load_package()
    peak, peak_src = measured_peak()
    info = dict(card(), hbm_peak_GBs=peak, hbm_peak_source=peak_src)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "decoder_train.jsonl")

    def emit(rec):
        rec.update(info)
        with open(path, "a") as f:
            f.write(json.dumps(rec) + "\n")
        print(json.dumps(rec), flush=True)
    parts = args.parts.split(",")
    if "a" in parts:
        part_a(pkg, args, emit, peak)
    if "b" in parts:
        part_b(pkg, args, emit)


if __name__ == "__main__":
    main()
