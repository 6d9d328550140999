"""Launch list of the pixel-decoder forward under bf16 autocast with linear="autocast" (torch.profiler, CUDA activity).

    python tools/prof_autocast_decoder.py [--out DIR] [--calls 5] [--linear autocast]

forward_features at the configs[2] shape (1024x2048, batch 8, Swin-T pyramid, 6 encoder layers, fused=True, amp=True),
no autograd, warmed up, then `--calls` profiled calls.  Writes DIR/decoder_launches.md: every kernel with its share of
the summed device time, time and launches per call.  The profiler slows the host, so the times here are shares; take
end-to-end times from tools/bench_mixed.py --parts b.
"""
import argparse
import collections
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from __graft_entry__ import load_package  # noqa: E402
from bench_decoder_train import card  # noqa: E402
from bench_mixed import _decoder, _feats  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.environ.get("BENCH_OUT") or os.path.join(ROOT, "bench_out"),
                                                  "mixed"))
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--linear", default="autocast")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("prof_autocast_decoder.py profiles on a CUDA device; none is available")
    pkg = load_package()
    m = _decoder(pkg, fused=True, linear=args.linear, amp=True, train=False)
    feats = _feats(8, 1024, 2048, 3)

    def fwd():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            m.forward_features(feats)
    for _ in range(3):
        fwd()
    torch.cuda.synchronize()
    acts = [torch.profiler.ProfilerActivity.CUDA]
    with torch.profiler.profile(activities=acts) as prof:
        for _ in range(args.calls):
            fwd()
        torch.cuda.synchronize()
    us, count = collections.Counter(), collections.Counter()
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            us[ev.name] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            count[ev.name] += 1
    total = sum(us.values())
    info = card()
    os.makedirs(args.out, exist_ok=True)
    lines = [f"# Pixel-decoder forward under bf16 autocast, linear=\"{args.linear}\", fused=True, amp=True",
             "",
             f"{info['gpu']}, power limit {info['power_limit']}; 1024x2048, batch 8, Swin-T pyramid, 6 encoder layers, "
             f"no autograd; torch.profiler (CUDA activity) over {args.calls} calls after 3 warm-up calls.",
             "",
             f"{sum(count.values())} launches, {total / 1e3:.1f} ms summed device time over {args.calls} calls = "
             f"{sum(count.values()) / args.calls:.0f} launches and {total / 1e3 / args.calls:.2f} ms per call",
             "",
             "| share | us per call | launches per call | kernel |",
             "|---:|---:|---:|---|"]
    for name, t in us.most_common():
        lines.append(f"| {100 * t / total:.1f} % | {t / args.calls:.0f} | {count[name] / args.calls:.1f} | "
                     f"`{name[:110]}` |")
    path = os.path.join(args.out, "decoder_launches.md")
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines[:40]))


if __name__ == "__main__":
    main()
