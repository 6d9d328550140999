#!/usr/bin/env python
"""bench.py -- MSDeformAttn forward+backward throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--mode model|uniform]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference's CPU path on the host cores

A "step" is one forward + one backward pass of the MSDA hot path over one synthetic batch
(default workload: BASELINE configs[1], the 512x1024 Cityscapes crop pyramid, batch 8 per GPU,
fp32).  Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.

Timing: per-step CUDA events on the launching stream; an untimed 512 MiB L2 flush between steps;
W >= 3 warm-up steps; max over ranks; SM clocks / throttle reasons sampled through NVML during
the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "msda_fwd_bwd_queries_per_s"
UNIT = "queries/s"
DEFAULT_WORKLOAD = "cityscapes_512x1024_b8"
NOMINAL_HBM_GBS = 8000.0          # north_star's "~8 TB/s"
# Counters of the dominant kernel that only a profiler can give (DRAM bytes, reduction sectors): read
# from the committed summary of the ncu --set full capture of THIS command for the current kernels
# (tools/ncu_counters.py writes it from the .ncu-rep; profiles/README.md).  A kernel the summary does
# not name gets null -- nothing here is pasted by hand.
NCU_COUNTERS_JSON = os.path.join(ROOT, "profiles", "r2_ncu_bench_counters.json")
L2_REDUCTION_GBS = 6400.0         # measured: profiles/r1_microbench.txt (red.global.add payload, chip-wide)
FALLBACK_HBM_GBS = 6650.0         # /opt/skills/guides/B200_PROFILING.md fallback


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=50,
                   help="timed steps of the measured metric (>= 1).  Two context figures of the GPU arm "
                        "keep their own counts, reported in the JSON line: the e2e leg times "
                        "max(4, min(K, 20)) steps, the CPU baseline 5")
    p.add_argument("--warmup", type=int, default=10)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--workload", default=DEFAULT_WORKLOAD)
    p.add_argument("--mode", default="model", choices=["model", "uniform"])
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--cpu-sample-batch", type=int, default=0,
                   help="images per CPU step; 0 = the workload's whole batch")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write rank 0's output and three gradients of the last "
                        "step as DIR/<name>.npy (float32); see dump_outputs()")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        p.error("--dump-outputs writes what the GPU arm computed; it needs --impl b200")
    return args


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.01)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ----------------------------------------------------------------------------- shared helpers
def load_synthetic():
    """uni-encoder-code_b200/synthetic.py imported BY PATH (plain torch, no CUDA library): the
    reference arm builds the same tensors as the GPU arm without ever loading libmsda_b200.so."""
    import importlib.util
    name = "msda_b200_synthetic"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "uni-encoder-code_b200", "synthetic.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def make_config(args, w):
    """Identical in both arms (the driver compares them key by key)."""
    return {
        "workload": f"{args.workload} fwd+bwd (BASELINE.json configs[1])",
        "levels": [list(x) for x in w.levels], "batch_per_gpu": w.batch, "heads": w.heads,
        "channels": w.channels, "points": w.points,
        "queries_per_step_per_gpu": w.batch * w.spatial_size, "loc_mode": args.mode,
        "l2": "512 MiB memset between steps (untimed); step working set 640 MB > 126 MB L2",
        "step": "forward + backward of the op on one batch, inputs resident in memory",
        "sharding": "batch (independent images per rank), no data-path collective",
    }


def ncu_counters(kernel_name, workload, mode):
    """{dram_bytes, red_sectors, ...} per launch for `kernel_name` from the committed capture, or {}."""
    try:
        with open(NCU_COUNTERS_JSON) as f:
            doc = json.load(f)
        if doc.get("workload") != workload or doc.get("mode") != mode:
            return {}
        return doc.get("kernels", {}).get(kernel_name, {})
    except Exception:
        return {}


# ----------------------------------------------------------------------------- CPU arms
def load_reference_core():
    """-> (function(value, shapes, loc, w) -> output, kind).

    kind "reference": the reference's OWN ms_deform_attn_core_pytorch, executed from the unmodified
    copy of ops/functions/ms_deform_attn_func.py that baseline/stage_reference_py.py stages under
    git-ignored baseline/_ref/py/ (it travels to the GPU box; /root/reference does not).  On a box
    with a GPU that file imports `MultiScaleDeformableAttention` when it is loaded (func.py:21-30);
    an empty stand-in module satisfies the import, so neither the repo's shim nor its CUDA library
    is touched -- the CPU function never uses it.
    kind "port": the restatement oracle.core_grid_sample, only when the staged file is absent."""
    import importlib.util
    import types
    path = os.path.join(ROOT, "baseline", "_ref", "py", "modeling", "pixel_decoder", "ops", "functions",
                        "ms_deform_attn_func.py")
    if os.path.isfile(path):
        had = sys.modules.get("MultiScaleDeformableAttention")
        if had is None:
            sys.modules["MultiScaleDeformableAttention"] = types.ModuleType("MultiScaleDeformableAttention")
        try:
            spec = importlib.util.spec_from_file_location("ref_ms_deform_attn_func", path)
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
        finally:
            if had is None:
                sys.modules.pop("MultiScaleDeformableAttention", None)
        return mod.ms_deform_attn_core_pytorch, "reference"
    from __graft_entry__ import load_oracle
    return load_oracle().core_grid_sample, "port"


def cpu_reference_run(workload_name, mode, sample_batch, steps, warmup):
    """The reference's CPU path for this op: ms_deform_attn_core_pytorch
    (ops/functions/ms_deform_attn_func.py:55-75) + autograd, fp32, on every host thread torch can
    use.  Each step is forward+backward on `sample_batch` images of the workload's shape."""
    import torch
    core, kind = load_reference_core()
    syn = load_synthetic()
    torch.set_num_threads(os.cpu_count() or 1)
    w = syn.WORKLOADS[workload_name]
    inp = syn.make_inputs(w.levels, sample_batch, w.heads, w.channels, w.points, mode=mode, seed=0)
    times = []
    for i in range(warmup + steps):
        v = inp["value"].detach().requires_grad_(True)
        loc = inp["sampling_locations"].detach().requires_grad_(True)
        wts = inp["attention_weights"].detach().requires_grad_(True)
        t0 = time.perf_counter()
        out = core(v, inp["spatial_shapes"], loc, wts)
        torch.autograd.grad(out, (v, loc, wts), inp["grad_output"])
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    q = sample_batch * w.spatial_size
    mean = sum(times) / len(times)
    what = ("the reference's ms_deform_attn_core_pytorch (staged unmodified file)" if kind == "reference"
            else "oracle.core_grid_sample (restated ms_deform_attn_core_pytorch)")
    return {"value": q / mean, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
            "host_cpus": os.cpu_count(),
            "sample": f"fwd+bwd (autograd) of {what}, fp32, on {sample_batch} image(s) of {workload_name} = "
                      f"{q} queries/step, {len(times)} timed steps after {warmup} warm-up",
            "ms_per_step": mean * 1e3}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = load_synthetic().WORKLOADS[args.workload]
    # the whole batch of the workload per step (~0.4-0.6 s on the host's cores): K is honoured, W is
    # capped at 5 warm-up steps
    steps = args.steps
    warmup = max(1, min(args.warmup, 5))
    batch = w.batch if args.cpu_sample_batch <= 0 else args.cpu_sample_batch
    base = cpu_reference_run(args.workload, args.mode, batch, steps, warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT,
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": base["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": make_config(args, w),
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm
def run_b200_arm(args):
    import torch
    import torch.distributed as dist
    from __graft_entry__ import load_package

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL_DEBUG is left as the caller set it: whatever NCCL prints on fd 1 goes to stderr (main())
        dist.init_process_group("nccl", device_id=dev)

    pkg = load_package()
    lib = pkg._lib.lib
    syn = pkg.synthetic
    w = syn.WORKLOADS[args.workload]
    # batch sharding (SURVEY 8e): every rank owns its own images; weak scaling, no data-path collective
    host = syn.make_inputs(w.levels, w.batch, w.heads, w.channels, w.points, mode=args.mode,
                           seed=1000 + rank)
    d = {k: v.to(dev) for k, v in host.items()}
    N, S, M, D = d["value"].shape
    L, Lq, P = len(w.levels), S, w.points
    out = torch.empty(N, Lq, M * D, device=dev)
    gv = torch.empty_like(d["value"])
    gl = torch.empty_like(d["sampling_locations"])
    gw = torch.empty_like(d["attention_weights"])
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()
    sp = stream.cuda_stream
    dims = (N, S, M, D, L, Lq, P)
    ptr = {k: v.data_ptr() for k, v in d.items()}

    def fwd():
        pkg._lib.check(lib.msda_b200_forward_f32(
            ptr["value"], ptr["spatial_shapes"], ptr["level_start_index"], ptr["sampling_locations"],
            ptr["attention_weights"], *dims, out.data_ptr(), sp), "forward")

    def bwd():
        pkg._lib.check(lib.msda_b200_backward_f32(
            ptr["grad_output"], ptr["value"], ptr["spatial_shapes"], ptr["level_start_index"],
            ptr["sampling_locations"], ptr["attention_weights"], *dims, gv.data_ptr(), gl.data_ptr(),
            gw.data_ptr(), sp), "backward")

    ev = lambda: torch.cuda.Event(enable_timing=True)
    marks = [[ev() for _ in range(4)] for _ in range(args.steps)]

    def step(m=None):
        flush.zero_()                       # untimed: evict inputs/outputs from the 126 MB L2
        if m: m[0].record(stream)
        fwd()
        if m: m[1].record(stream)
        gv.zero_()                          # grad_value is accumulated with reductions
        if m: m[2].record(stream)
        bwd()
        if m: m[3].record(stream)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    n0 = pkg.launch_count()
    with ClockSampler(local_rank) as clocks:
        t_wall0 = time.perf_counter()
        for i in range(args.steps):
            step(marks[i])
        torch.cuda.synchronize()
        t_wall = time.perf_counter() - t_wall0
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches = pkg.launch_count() - n0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"output": out, "grad_value": gv, "grad_sampling_loc": gl,
                                         "grad_attn_weight": gw})

    step_ms = [m[0].elapsed_time(m[3]) for m in marks]
    fwd_ms = [m[0].elapsed_time(m[1]) for m in marks]
    zero_ms = [m[1].elapsed_time(m[2]) for m in marks]
    bwd_ms = [m[2].elapsed_time(m[3]) for m in marks]
    total_ms = sum(step_ms)
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    queries_rank = N * Lq
    ms_per_step = total_ms / args.steps
    value = world * queries_rank / (ms_per_step * 1e-3)

    # ---- end to end through the plugin API with host buffers (rank-local, then max over ranks)
    e2e = None
    if not args.no_e2e:
        old_affinity = bind_near_gpu(local_rank)
        e2e = run_e2e(pkg, host, dev, world, max(4, min(args.steps, 20)), dist if world > 1 else None)
        e2e["cpus_bound"] = len(os.sched_getaffinity(0))
        if old_affinity:
            os.sched_setaffinity(0, old_affinity)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak()
    bwd_mean = statistics.mean(bwd_ms)
    fwd_mean = statistics.mean(fwd_ms)
    bwd_bytes = queries_rank * syn.BWD_BYTES_PER_QUERY
    fwd_bytes = queries_rank * syn.FWD_BYTES_PER_QUERY
    achieved = bwd_bytes / (bwd_mean * 1e-3) / 1e9
    # which backward kernel the library's location probe picked for these inputs (model-like
    # locations: the in-SM merging kernel; uniform ones: the per-row reduction kernel)
    bwd_kernel = "msda_bwd_sorted_kernel" if args.mode == "model" else "msda_bwd_d32_kernel"
    ctr = ncu_counters(bwd_kernel, args.workload, args.mode)
    red_bytes = ctr.get("red_sectors", 0) * 32
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(args, w),
        "roofline": {
            "bound": "hbm", "kernel": bwd_kernel, "achieved": achieved, "peak": peak,
            "unit": "GB/s", "frac": achieved / peak,
            "traffic": ctr.get("dram_bytes"),
            "traffic_source": ("profiles/r2_ncu_bench_counters.json (ncu --set full of this command, per launch)"
                               if ctr else "no committed capture names this kernel: see profiles/"),
            "peak_source": peak_src,
            "algorithmic_bytes_per_launch": bwd_bytes, "ms_per_launch": bwd_mean,
            "timed": "CUDA events around msda_b200_backward_f32 (location probe + the chosen kernel), "
                     "mean over the timed steps",
            "frac_of_nominal_8TBs": achieved / NOMINAL_HBM_GBS,
            "on_chip_limiter": ({
                "resource": "L2 reduction (red.global.add) payload",
                "bytes_per_launch": red_bytes,
                "achieved_GBs": red_bytes / (bwd_mean * 1e-3) / 1e9,
                "measured_peak_GBs": L2_REDUCTION_GBS,
                "frac": red_bytes / (bwd_mean * 1e-3) / 1e9 / L2_REDUCTION_GBS,
                "l1_data_pipe_pct": ctr.get("l1_data_pipe_pct"),
                "issue_slot_pct": ctr.get("issue_active_pct"),
                "source": "profiles/r2_ncu_bench_counters.json, profiles/r1_microbench.txt; DESIGN.md section 4",
            } if ctr else None),
        },
        "kernels": {
            "forward": {"ms": fwd_mean, "algorithmic_GBs": fwd_bytes / (fwd_mean * 1e-3) / 1e9,
                        "frac": fwd_bytes / (fwd_mean * 1e-3) / 1e9 / peak},
            "grad_value_memset": {"ms": statistics.mean(zero_ms)},
            "backward": {"ms": bwd_mean, "algorithmic_GBs": achieved, "frac": achieved / peak,
                         "kernel": bwd_kernel},
            "fwd_bwd": {"algorithmic_GBs": (fwd_bytes + bwd_bytes) / (ms_per_step * 1e-3) / 1e9,
                        "frac": (fwd_bytes + bwd_bytes) / (ms_per_step * 1e-3) / 1e9 / peak},
        },
        "gpu_launches": launches,
        "clocks": clocks.summary(),
        "wall_ms_per_step_incl_flush": t_wall / args.steps * 1e3,
    }
    if e2e is not None:
        line["e2e"] = e2e
    if world == 1:
        ref_cuda = reference_cuda_same_gpu(pkg, d, flush)
        if ref_cuda is not None:
            line["reference_cuda_same_gpu"] = ref_cuda
    if world == 1 and not args.no_cpu_baseline:
        batch = w.batch if args.cpu_sample_batch <= 0 else args.cpu_sample_batch
        base = cpu_reference_run(args.workload, args.mode, batch, 5, 1)
        line["cpu_baseline"] = {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 60 << 20      # keeps the .npy files of --dump-outputs, headers included, under 64 MB


def dump_outputs(directory, arrays, seed=0):
    """Write each [N, S, ...] device tensor of `arrays` as <directory>/<name>.npy in float32, flattened to
    [rows, ...] with one row per (image, query).  When all rows of all tensors exceed DUMP_BYTES, every
    tensor keeps the same rows: a sample drawn with a fixed seed, in ascending order.  The inputs of a
    run depend only on its arguments, so two builds run alike write files that compare element by element."""
    import numpy as np
    import torch
    rows = {t.shape[0] * t.shape[1] for t in arrays.values()}
    assert len(rows) == 1, "every dumped tensor has one row per (image, query)"
    rows = rows.pop()
    row_bytes = sum(t[0, 0].numel() * 4 for t in arrays.values())
    keep = min(rows, DUMP_BYTES // row_bytes)
    idx = None
    if keep < rows:
        pick = np.sort(np.random.default_rng(seed).choice(rows, keep, replace=False))
        idx = torch.from_numpy(pick).to(next(iter(arrays.values())).device)
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        flat = t.detach().reshape(rows, *t.shape[2:])
        if idx is not None:
            flat = flat.index_select(0, idx)
        np.save(os.path.join(directory, name + ".npy"), flat.float().cpu().numpy())


def reference_cuda_same_gpu(pkg, d, flush, iters=5):
    """Context only (not an arm): the reference's own CUDA op, compiled for sm_100 in the build
    container by baseline/build_reference_cuda.py, timed on the same tensors when its .so travelled."""
    import importlib.util
    import torch
    so = os.path.join(ROOT, "baseline", "_ref", "ref_msda_cuda.so")
    if not os.path.exists(so):
        return None
    try:
        spec = importlib.util.spec_from_file_location("ref_msda_cuda", so)
        ref = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(ref)
        a = (d["value"], d["spatial_shapes"], d["level_start_index"], d["sampling_locations"],
             d["attention_weights"])

        def t(fn):
            ts = []
            for i in range(2 + iters):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                if i >= 2:
                    ts.append(e0.elapsed_time(e1))
            return sum(ts) / len(ts)
        f = t(lambda: ref.ms_deform_attn_forward(*a, 128))
        b = t(lambda: ref.ms_deform_attn_backward(*a, d["grad_output"], 128))
        q = d["value"].shape[0] * d["sampling_locations"].shape[1]
        return {"forward_ms": f, "backward_ms": b, "queries_per_s": q / ((f + b) * 1e-3),
                "what": "reference ms_deform_attn_forward/backward (its CUDA kernels, sm_100 build) per call "
                        "incl. its own zero-fills; see profiles/r1_vs_reference_cuda.md"}
    except Exception as e:      # a comparison aid must never break the bench line
        return {"unavailable": repr(e)[:200]}


def bind_near_gpu(index):
    """Pin this process to the CPUs NVML reports as local to GPU `index` (intersected with what the
    container allows), so the pinned host buffers of the e2e leg are first-touched on the GPU's NUMA
    node.  Returns the previous affinity (restored before the CPU baseline uses every core)."""
    try:
        import pynvml
        before = os.sched_getaffinity(0)
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (max(before) // 64) + 1)
        near = {i * 64 + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        pick = near & before
        if pick and pick != before:
            os.sched_setaffinity(0, pick)
        return before
    except Exception:
        return None


def run_e2e(pkg, host, dev, world, steps, dist):
    """Same metric through the public plugin call (MSDeformAttnFunction.apply + autograd backward)
    with HOST buffers: every step copies its inputs from pinned host memory to the device and the
    four results back to pinned host memory, all inside the timed region.

    The three legs run on three streams with double-buffered device inputs and host outputs, so
    the H2D copy of step i+1, the kernels of step i and the D2H copy of step i-1 overlap (PCIe is
    full duplex); per-step work is unchanged."""
    import torch
    pin = {k: v.pin_memory() for k, v in host.items()}
    names = list(pin)
    cur = torch.cuda.current_stream()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    dev_in = [{k: torch.empty_like(v, device=dev) for k, v in pin.items()} for _ in range(2)]
    in_ready = [torch.cuda.Event() for _ in range(2)]
    in_free = [torch.cuda.Event() for _ in range(2)]
    out_done = [torch.cuda.Event() for _ in range(2)]
    res_host = [None, None]
    h2d = sum(v.numel() * v.element_size() for v in pin.values())
    d2h = 0

    def one(i):
        nonlocal d2h
        b = i & 1
        with torch.cuda.stream(s_in):
            s_in.wait_event(in_free[b])                 # kernels of step i-2 no longer read buffer b
            for k in names:
                dev_in[b][k].copy_(pin[k], non_blocking=True)
            in_ready[b].record(s_in)
        cur.wait_event(in_ready[b])
        d = dev_in[b]
        value = d["value"].detach().requires_grad_(True)
        loc = d["sampling_locations"].detach().requires_grad_(True)
        wts = d["attention_weights"].detach().requires_grad_(True)
        out = pkg.MSDeformAttnFunction.apply(value, d["spatial_shapes"], d["level_start_index"],
                                             loc, wts, 128)
        grads = torch.autograd.grad(out, (value, loc, wts), d["grad_output"])
        in_free[b].record(cur)
        results = (out.detach(),) + tuple(grads)
        if res_host[b] is None:
            res_host[b] = [torch.empty(r.shape, dtype=r.dtype, pin_memory=True) for r in results]
            d2h = sum(r.numel() * r.element_size() for r in results)
        done = torch.cuda.Event()
        done.record(cur)
        with torch.cuda.stream(s_out):
            s_out.wait_event(done)
            s_out.wait_event(out_done[b])               # host buffer b of step i-2 is complete
            for h, r in zip(res_host[b], results):
                h.copy_(r, non_blocking=True)
                r.record_stream(s_out)
            out_done[b].record(s_out)

    # warm-up: first-touch of the pinned buffers, allocator pools, and the PCIe link leaving its idle
    # state (the first transfers of a fresh process were measured ~40 % slower)
    for i in range(16):
        one(i)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    # the host side (pinned memory, PCIe root) is shared with other tenants of the box: three
    # repetitions of `steps` steps, the MEDIAN is reported and all three are listed
    trials = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(cur)
        for i in range(steps):
            one(i)
        cur.wait_stream(s_out)
        cur.wait_stream(s_in)
        e1.record(cur)
        torch.cuda.synchronize()
        trials.append(e0.elapsed_time(e1))
    ms = statistics.median(trials)
    if dist is not None:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    q = host["value"].shape[0] * host["sampling_locations"].shape[1]
    return {"value": world * q * steps / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "ms_per_step": ms / steps, "steps": steps,
            "trials_ms_per_step": [t / steps for t in trials],
            "api": "MSDeformAttnFunction.apply + autograd.grad; pinned host -> device inputs and "
                   "device -> pinned host results every step, copies overlapped with compute on "
                   "3 streams (double-buffered); median of 3 repetitions of `steps` steps"}


def main():
    args = parse_args()
    # stdout carries exactly ONE JSON line: anything libraries print on fd 1 while the run is in
    # progress (e.g. NCCL's version banner at communicator creation) is sent to stderr instead
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    line_holder = []
    real_print = print

    def capture(*a, **k):
        line_holder.append(" ".join(str(x) for x in a))
    globals()["print"] = capture
    try:
        if args.impl == "reference":
            run_reference_arm(args)
        else:
            run_b200_arm(args)
    finally:
        globals()["print"] = real_print
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
    for line in line_holder:
        real_print(line, flush=True)


if __name__ == "__main__":
    main()
