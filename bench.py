#!/usr/bin/env python
"""MSDeformAttn hot-path benchmark (driver contract: one JSON line on stdout from rank 0).

  python bench.py --gpus N --steps K --warmup W            # the sm_100a kernels
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port)
  python bench.py ... --dump-outputs DIR                   # also save what the last timed step computed

The K timed steps are split into --regions regions (default 3); the reported step time is the median region's.

Metric (BASELINE.json): sampled-points/s of MSDeformAttn forward+backward, point = one
(b,q,h,l,p) sample.  Workload at any N: BASELINE configs[1] per GPU -- the DINO-R50 deformable
encoder's self-attention, 6 layers, batch 8 @ 800x1333 (levels 100x167, 50x84, 25x42, 13x21,
Q = S = 22223, 8 heads x 32 channels, 4 points), fp32.  One STEP = the core op's forward and
backward for all 6 layers (6 distinct input sets, ~1.3 GB each, so nothing survives in the 126 MB
L2 between uses).  N > 1 shards by image batch (weak scaling, 8 images per GPU, no collective
inside the op; nothing is exchanged).  `--scaling strong --total-batch N` splits a fixed batch over the
GPUs; `--mode train` is BASELINE config 4, the batch-sharded training step: 6 MSDeformAttn modules forward +
backward, per-module NCCL all-reduce of the projection-weight gradients launched from gradient hooks, fused AdamW.

  value     points/s with inputs resident in HBM, CUDA-event timed, max over ranks
  e2e       the same through the public autograd API with HOST buffers: pinned host -> device copies
            of value / locations / weights / grad_output and device -> host copies of the output
            and the three gradients inside the timed region
  roofline  dominant kernel (backward): algorithmic bytes per launch / its mean CUDA-event
            duration, against MEASURED_PEAKS.json hbm_gbs (fallback 6650 GB/s)
  cpu_baseline  oracle/msda_torch (the reference's grid_sample formulation) on the host cores,
            bounded sample (one encoder layer at B=1), rank 0 only
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from ir_ads_b200.workloads import WORKLOADS, make_workload_inputs  # noqa: E402

NUM_LAYERS = 6
METRIC = "msda_fwd_bwd_sampled_points_per_s"
UNIT = "points/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--dist", default="model", choices=["model", "test", "edge"])
    ap.add_argument("--layers", type=int, default=NUM_LAYERS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true")
    ap.add_argument("--flags", type=int, default=0, help="extra MSDA_FLAG_* bits (experiments)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the workload's batch per GPU; strong: --total-batch images split over the GPUs")
    ap.add_argument("--total-batch", type=int, default=0, help="strong scaling: images in the whole job")
    ap.add_argument("--mode", default="op", choices=["op", "train"],
                    help="op: the core operator (the metric); train: batch-sharded module-level training step "
                         "(projections + fused op, fwd+bwd, grad all-reduce overlapped with backward, optimizer)")
    ap.add_argument("--regions", type=int, default=3,
                    help="timed regions the --steps timed steps are split into (median per-step time reported)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="op mode: write what the last timed step computed (out and the three gradients of every layer, "
                         "float32, a fixed seeded sample of each large tensor, under 64 MB in all) as DIR/<name>.npy.  That "
                         "step keeps its outputs alive, so the allocator may have to allocate inside the last timed region")
    ap.add_argument("--no-graph", action="store_true", help="train mode: do not try CUDA-graph capture")
    ap.add_argument("--amp", action="store_true", help="train mode: bf16 autocast (AMP config)")
    ap.add_argument("--tf32", action="store_true",
                    help="train mode: TF32 tensor-core matmuls for the fp32 projections (torch 1.10, which the reference "
                         "pins, enabled them by default; torch 2.x does not)")
    return ap.parse_args()


def config_dict(wl, args, extra=None):
    cfg = {
        "workload": f"{wl.name}: DINO-R50 deformable encoder self-attn core op fwd+bwd, {args.layers} layers"
        if wl.name == "cfg2" else f"{wl.name} core op fwd+bwd, {args.layers} layers",
        "levels": [list(x) for x in wl.levels], "batch_per_gpu": wl.batch, "num_query": wl.queries,
        "heads": wl.num_heads, "head_dim": wl.head_dim, "points": wl.num_points, "value_dtype": wl.value_dtype,
        "points_per_step_per_gpu": wl.points * args.layers, "dist": args.dist,
        "l2_hygiene": f"{args.layers} distinct layer input sets cycled per step "
                      f"({wl.algorithmic_bytes()[0] / 1e6:.0f} MB of inputs each"
                      f"{', larger than the 126 MB L2' if wl.batch >= 4 else '; plus an L2 flush (256 MB write) between timed regions'})",
        "parallelism": f"image-batch sharding x{args.gpus}, no collective inside or around the core op (NCCL: barrier and "
                       "max-over-ranks of the step time only; the training config's gradient all-reduce is in --mode train)",
        "scaling_mode": args.scaling, "total_batch": wl.batch * args.gpus,
    }
    if extra:
        cfg.update(extra)
    return cfg


def split_steps(steps, regions):
    """The `steps` timed steps split as evenly as possible into up to `regions` timed regions."""
    n = max(1, min(regions, steps))
    return [steps // n + (r < steps % n) for r in range(n)]


# --------------------------------------------------------------------------------------------
# clocks sampling (NVML; nvidia-smi fallback)
# --------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting",
               0x10: "sync_boost"}

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nvml = None

    def _loop(self):
        nv = self._nvml
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def _smi_loop(self):
        """Fallback when NVML's python binding is missing: poll nvidia-smi (B200_PROFILING.md's clocks line)."""
        import subprocess
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append(int(f[0]))
                self.max_mhz = int(f[1])
                for name, val in zip(names, f[2:]):
                    if val.lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.05)

    def start(self):
        target = self._loop if self._nvml is not None else self._smi_loop
        self._thread = threading.Thread(target=target, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------
# CPU baseline (oracle port): rank 0 only, bounded sample
# --------------------------------------------------------------------------------------------
def cpu_baseline(wl, dist, iters=40, budget_s=15.0):
    from oracle import msda_torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    value, shapes, lsi, loc, w = make_workload_inputs(wl, dist, seed=0, device="cpu", batch=1)
    value = value.float()
    go = torch.randn(1, wl.queries, wl.num_heads * wl.head_dim)
    pts = wl.points // wl.batch
    msda_torch.forward_backward(value, shapes, loc, w, go)          # warm-up
    times = []
    t_start = time.perf_counter()
    for _ in range(iters):
        t0 = time.perf_counter()
        msda_torch.forward_backward(value, shapes, loc, w, go)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s:
            break
    t = statistics.median(times)
    return {"value": pts / t, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"one layer of {wl.name} at batch 1 ({pts} points), fwd + autograd bwd, fp32, "
                      f"median of {len(times)} after 1 warm-up, {t * 1e3:.0f} ms each"}


def run_reference_arm(args, wl):
    """--impl reference: the reference's CPU path (oracle port of multi_scale_deformable_attn_pytorch)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import msda_torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    value, shapes, lsi, loc, w = make_workload_inputs(wl, args.dist, seed=0, device="cpu", batch=1)
    value = value.float()
    Q = wl.queries
    go = torch.randn(1, Q, wl.num_heads * wl.head_dim)
    t0 = time.perf_counter()
    msda_torch.forward_backward(value, shapes, loc, w, go)
    probe = time.perf_counter() - t0
    # bounded sample: keep the whole run (warm-up + steps) under ~3 minutes by taking a query prefix
    total_iters = args.steps + args.warmup
    frac = min(1.0, 170.0 / max(probe * total_iters, 1e-9))
    q_used = max(64, int(Q * frac))
    loc, w, go = loc[:, :q_used].contiguous(), w[:, :q_used].contiguous(), go[:, :q_used].contiguous()
    pts = q_used * wl.num_heads * wl.num_levels * wl.num_points
    for _ in range(args.warmup):
        msda_torch.forward_backward(value, shapes, loc, w, go)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        msda_torch.forward_backward(value, shapes, loc, w, go)
    dt = time.perf_counter() - t0
    val = pts * args.steps / dt
    sample = (f"one layer of {wl.name} at batch 1, first {q_used} of {Q} queries ({pts} points per step), "
              f"fwd + autograd bwd, fp32, torch {torch.__version__}")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(wl, args, {"reference_sample": sample}),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# the B200 arm
# --------------------------------------------------------------------------------------------
def peak_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(workload: str, kernel: str):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/ncu_traffic.json), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)[workload].get(kernel)
    except Exception:
        return None


def onchip_block(wl, fwd_ms, bwd_ms, valid_frac):
    """The measured on-chip ceilings (profiles/microbench_ceilings.json) scaled to the corner rows this workload
    actually moves: the kernels gather up to 4 corner rows of D channels per point through L1 and scatter as many
    through L2 reds (padded corners -- `valid_frac` of the 4 * N are inside their level -- are neither loaded nor
    scattered); those rates, not HBM, bound them (DESIGN.md section 6).  Reported beside the HBM fraction, never
    instead of it."""
    try:
        with open(os.path.join(ROOT, "profiles", "microbench_ceilings.json")) as f:
            c = json.load(f)
    except Exception:
        return None
    if wl.value_dtype != "f32" or wl.head_dim != 32:
        return None                                  # the ceilings were measured on 128-byte float rows
    rows = wl.points * 4
    k = rows * valid_frac / c["rows_measured"]
    g1, g2, red = c["gather_l1_resident_ms"] * k, c["gather_l2_sourced_ms"] * k, c["red_v4_f32_l2_resident_ms"] * k
    return {"corner_rows_per_launch": rows, "corner_rows_inside_the_map": int(rows * valid_frac), "row_bytes": c["row_bytes"],
            "ceilings_ms": {"fwd_gather_l1_resident": g1, "fwd_gather_l2_sourced": g2, "bwd_red_l2_rate": red},
            "fwd_frac_of_onchip_ceiling": g2 / fwd_ms, "bwd_frac_of_onchip_ceiling": red / bwd_ms,
            "ncu_counters_cfg2": c.get("ncu_counters_cfg2"),
            "note": "ceiling for the rows inside the map / measured launch time (backward: incl. its grad_value zero-fill)",
            "source": "profiles/microbench_ceilings.json (tools/microbench/*.cu on this pool's B200s)"}


def main():
    args = parse_args()
    wl = WORKLOADS[args.workload]
    if args.steps < 1:
        raise SystemExit("bench.py: --steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.mode != "op"):
        raise SystemExit("bench.py: --dump-outputs covers the sm_100a core op (--impl b200 --mode op) only")
    if args.impl == "reference":
        run_reference_arm(args, wl)
        return

    import dataclasses

    import ir_ads_b200
    from ir_ads_b200 import _lib, functional

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist_on = world > 1
    if dist_on:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    args.gpus = world
    if args.scaling == "strong":
        from ir_ads_b200.sharding import shard_batch
        total = args.total_batch or wl.batch
        _, per = shard_batch(total, world, rank)          # raises unless the batch divides evenly
        wl = dataclasses.replace(wl, batch=per)
    if args.mode == "train":
        run_train_mode(args, wl, dev, rank, world, dist_on)
        if dist_on:
            dist.barrier()
            dist.destroy_process_group()
        return

    L = args.layers
    n_pts_layer = wl.points
    fwd_bytes, bwd_bytes = wl.algorithmic_bytes()
    out_dt = torch.bfloat16 if wl.value_dtype == "bf16" else torch.float32
    if wl.deterministic:
        functional.set_deterministic(True)

    layers = []
    for i in range(L):
        value, shapes, lsi, loc, w = make_workload_inputs(wl, args.dist, seed=100 * rank + i, device=dev)
        go = torch.randn(wl.batch, wl.queries, wl.num_heads * wl.head_dim, device=dev,
                         generator=torch.Generator(device=dev).manual_seed(7 + i)).to(out_dt)
        layers.append((value, shapes, lsi, loc, w, go))
    # small per-GPU batches (strong scaling) fit in L2: flush it between timed regions
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if wl.batch < 4 else None
    # No collective in this mode: the core operator shards by image and exchanges nothing (SURVEY section 8e).  The
    # training config's gradient all-reduce is measured where real gradients exist: --mode train.
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def step(record=None, keep=False):
        """One step over all layers; with `keep`, returns every layer's (out, grad_value, grad_loc, grad_w)."""
        kept = []
        for i, (value, shapes, lsi, loc, w, go) in enumerate(layers):
            if record is not None:
                e0, e1, e2 = ev(), ev(), ev()
                e0.record()
            out = ir_ads_b200.ms_deform_attn_forward(value, shapes, lsi, loc, w, 64)
            if record is not None:
                e1.record()
            grads = ir_ads_b200.ms_deform_attn_backward(value, shapes, lsi, loc, w, go, 64)
            if record is not None:
                e2.record()
                record.append((e0, e1, e2))
            if keep:
                kept.append((out, *grads))
            del out, grads
        return kept

    def barrier():
        if dist_on:
            dist.barrier()
        torch.cuda.synchronize()

    with functional.kernel_flags(args.flags):
        for _ in range(max(args.warmup, 3)):
            step()
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        # the `steps` timed steps are split into up to `regions` timed regions, every one bracketed by barrier +
        # synchronize; the median region's per-step time is the reported one (one un-repeated sample gave an
        # unexplained 0.90 outlier in r01)
        region_steps = split_steps(args.steps, args.regions)
        n_regions = len(region_steps)
        region_ms = []
        launches = 0
        last = None
        for r, n in enumerate(region_steps):
            if flush is not None:
                flush.zero_()
            barrier()
            launches0 = _lib.launch_count()
            t_begin, t_end = ev(), ev()
            t_begin.record()
            for s in range(n):
                last = step(keep=bool(args.dump_outputs) and r == n_regions - 1 and s == n - 1)
            t_end.record()
            barrier()
            launches += _lib.launch_count() - launches0
            region_ms.append(t_begin.elapsed_time(t_end) / n)
        clocks = sampler.stop()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, last)
        del last

        # per-kernel durations (same stream, separate short pass so event records do not perturb `value`)
        recs = []
        for _ in range(3):
            step(recs)
        torch.cuda.synchronize()
        fwd_ms = statistics.median(a.elapsed_time(b) for a, b, _ in recs)
        bwd_ms = statistics.median(b.elapsed_time(c) for _, b, c in recs)

    if dist_on:
        from ir_ads_b200.sharding import max_over_ranks
        region_ms = [max_over_ranks(x, dev) for x in region_ms]
    ms_step = statistics.median(region_ms)
    value_pts = n_pts_layer * L * world / (ms_step * 1e-3)

    # ---------------- e2e: public autograd API, host buffers ----------------
    e2e = None
    if not args.no_e2e:
        with functional.kernel_flags(args.flags):
            e2e = run_e2e(wl, layers, dev, dist_on, world, args)

    ref_cuda = None
    if rank == 0 and not args.no_ref_cuda and wl.value_dtype == "f32":
        ref_cuda = run_ref_cuda(layers[:3], n_pts_layer)

    if rank == 0:
        peak, peak_src = peak_hbm()
        achieved = bwd_bytes / (bwd_ms * 1e-3) / 1e9
        flags_eff = args.flags | (_lib.FLAG_DETERMINISTIC if wl.deterministic else 0)
        bwd_name = _lib.lib().msda_dispatch_name(
            wl.head_dim, wl.num_levels, wl.num_points, wl.spatial_size, wl.num_heads,
            _lib.MSDA_BF16 if wl.value_dtype == "bf16" else _lib.MSDA_F32, flags_eff, 1).decode()
        if wl.deterministic:
            bwd_name += " (MSDA_FLAG_DETERMINISTIC: sorted segment reduction, several launches)"
        roof = {"bound": "hbm", "kernel": bwd_name,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "frac_of_nominal_8TBs": achieved / 8000.0,
                "traffic": ncu_traffic(wl.name, bwd_name) if args.flags == 0 and wl.batch == WORKLOADS[wl.name].batch else None,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": bwd_bytes,
                "launch_ms": bwd_ms, "note": "launch_ms includes the grad_value zero-fill memset issued by msda_backward",
                "fwd": {"algorithmic_bytes_per_launch": fwd_bytes, "launch_ms": fwd_ms,
                        "achieved": fwd_bytes / (fwd_ms * 1e-3) / 1e9, "frac": fwd_bytes / (fwd_ms * 1e-3) / 1e9 / peak},
                "fwd_bwd_frac": (fwd_bytes + bwd_bytes) / ((fwd_ms + bwd_ms) * 1e-3) / 1e9 / peak}
        from ir_ads_b200.workloads import valid_corner_fraction
        oc = onchip_block(wl, fwd_ms, bwd_ms, valid_corner_fraction(layers[0][3], wl.levels)) if not wl.deterministic else None
        if oc is not None:
            roof["onchip"] = oc
        line = {
            "metric": METRIC, "value": value_pts, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32" if wl.value_dtype == "f32" else "bf16(value) + f32 accumulate",
            "data": "synthetic", "config": config_dict(wl, args),
            "timed_regions": {"count": len(region_ms), "steps": region_steps, "ms_per_step": [round(x, 4) for x in region_ms],
                              "reported": "median", "spread_pct": round(100.0 * (max(region_ms) - min(region_ms)) / ms_step, 2)},
            "roofline": roof,
            "gpu_launches": int(launches), "clocks": clocks,
        }
        if e2e is not None:
            line["e2e"] = e2e
        if ref_cuda is not None:
            line["reference_cuda_same_gpu"] = ref_cuda
        if not args.no_cpu_baseline and world >= 1:
            line["cpu_baseline"] = cpu_baseline(WORKLOADS[args.workload], args.dist)
        print(json.dumps(line), flush=True)
    if dist_on:
        dist.barrier()
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------
# --mode train: BASELINE config 4, the batch-sharded deformable-DETR training step
# --------------------------------------------------------------------------------------------
def run_train_mode(args, wl, dev, rank, world, dist_on):
    """One step = `layers` MultiScaleDeformableAttention MODULES chained (value/offset/weight/output projections through
    cuBLAS, softmax + location affine + core op fused in the sm_100a kernels), forward + backward, the DDP-style mean
    all-reduce of the projection-weight gradients launched per module from gradient hooks so that it overlaps the rest of
    the backward (detectron2/detectron2/engine/defaults.py:60-79 wraps the model in DistributedDataParallel, whose
    buckets do the same), and a fused AdamW step.  Images are sharded over the ranks (total batch fixed under --scaling
    strong); no collective inside the op.  The step is replayed from one CUDA graph when capture succeeds."""
    import torch.distributed as dist
    from ir_ads_b200 import MultiScaleDeformableAttention, _lib, sharding
    from ir_ads_b200.workloads import _pixel_centres, level_tensors

    L = args.layers
    E = wl.num_heads * wl.head_dim
    if args.tf32:
        torch.backends.cuda.matmul.allow_tf32 = True
    torch.manual_seed(0)                                    # identical initial weights on every rank (DDP broadcast)
    mods = torch.nn.ModuleList([MultiScaleDeformableAttention(E, wl.num_heads, wl.num_levels, wl.num_points, dropout=0.0,
                                                              batch_first=True) for _ in range(L)]).to(dev)
    for m in mods:
        with torch.no_grad():                               # data-dependent offsets / weights, as after some training
            m.sampling_offsets.weight.normal_(0, 0.02)
            m.attention_weights.weight.normal_(0, 0.1)
    params = sharding.projection_parameters(mods)
    sync = sharding.OverlappedGradSync([sharding.projection_parameters([m]) for m in mods])
    opt = torch.optim.AdamW(params, lr=1e-5, fused=True, capturable=True)
    shapes, lsi = level_tensors(wl.levels, dev)
    level_shapes = list(wl.levels)
    S = wl.spatial_size
    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    x = torch.randn(wl.batch, S, E, device=dev, generator=g)
    pos = torch.randn(wl.batch, S, E, device=dev, generator=g) * 0.1
    ref = _pixel_centres(wl.levels, dev)[None, :, None, :].expand(wl.batch, S, wl.num_levels, 2).contiguous()
    amp = torch.autocast("cuda", dtype=torch.bfloat16) if args.amp else contextlib.nullcontext()

    def fwd_bwd():
        sync.zero_()
        with amp:
            h = x
            for m in mods:
                h = m(h, query_pos=pos, reference_points=ref, spatial_shapes=shapes, level_start_index=lsi,
                      level_shapes=level_shapes)
            loss = h.float().square().mean()
        loss.backward()                                     # hooks launch the per-module all-reduces as grads land
        sync.finish()
        opt.step()
        return loss

    def barrier():
        if dist_on:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(3):
        fwd_bwd()
    barrier()
    graph, how = None, "eager"
    if not args.no_graph:
        try:
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                fwd_bwd()
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_loss = fwd_bwd()
            graph.replay()
            torch.cuda.synchronize()
            how = "one CUDA graph per step (forward, backward, all-reduces, AdamW)"
        except Exception as exc:                            # capture of NCCL work is not guaranteed everywhere
            graph = None
            how = f"eager (graph capture failed: {type(exc).__name__})"
            torch.cuda.synchronize()
    step = graph.replay if graph is not None else fwd_bwd
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    region_steps = split_steps(args.steps, args.regions)
    region_ms = []
    launches = 0
    ev = lambda: torch.cuda.Event(enable_timing=True)
    for n in region_steps:
        flush.zero_()
        barrier()
        l0 = _lib.launch_count()
        t0, t1 = ev(), ev()
        t0.record()
        for _ in range(n):
            step()
        t1.record()
        barrier()
        launches += _lib.launch_count() - l0
        region_ms.append(t0.elapsed_time(t1) / n)
    clocks = sampler.stop()
    if dist_on:
        region_ms = [sharding.max_over_ranks(v, dev) for v in region_ms]
    ms = statistics.median(region_ms)
    pts = wl.points * L * world
    if rank == 0:
        kernels_per_step = 2 * L                            # fused forward + fused backward per module
        line = {
            "metric": "msda_training_step_sampled_points_per_s", "value": pts / (ms * 1e-3), "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "bf16 autocast (bf16 value, f32 accumulate)" if args.amp else
                     ("f32 (projections: TF32 tensor-core matmul)" if args.tf32 else "f32"), "data": "synthetic",
            "config": {"workload": f"{wl.name}: batch-sharded deformable-DETR training step -- {L} MSDeformAttn modules "
                                   "(projections + fused core op) fwd+bwd, per-module NCCL mean all-reduce of the "
                                   "projection-weight grads from gradient hooks, fused AdamW",
                       "levels": [list(v) for v in wl.levels], "batch_per_gpu": wl.batch, "total_batch": wl.batch * world,
                       "num_query": wl.queries, "heads": wl.num_heads, "head_dim": wl.head_dim, "points": wl.num_points,
                       "params_exchanged": sum(p.numel() for p in params), "execution": how,
                       "l2_hygiene": "256 MB L2 flush between timed regions",
                       "parallelism": f"image-batch sharding x{world}, no collective inside the op; "
                                      f"{L} all-reduces of 0.92 MB per step overlapped with backward"},
            "timed_regions": {"count": len(region_ms), "steps": region_steps, "ms_per_step": [round(v, 4) for v in region_ms],
                              "reported": "median", "spread_pct": round(100.0 * (max(region_ms) - min(region_ms)) / ms, 2)},
            "gpu_launches": int(launches) if graph is None else kernels_per_step * args.steps,
            "gpu_launches_note": "graph replays launch the captured kernels without passing the library's counter"
                                 if graph is not None else "counted by the library",
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)


DUMP_BYTES = 60 << 20      # the whole dump, float32 (under 64 MB with the .npy headers)


def dump_outputs(path, results):
    """Save each layer's forward output and its three gradients as float32 `layer<i>_<name>.npy` under `path`.  A tensor
    of more than DUMP_BYTES / (4 tensors x layers x 4 bytes) elements is reduced to that many elements at flat indices
    drawn from a fixed seed (sorted), the same for every run and build, so that two builds can be compared element for
    element."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    sample = DUMP_BYTES // (4 * 4 * max(1, len(results)))
    index = {}
    for i, tensors in enumerate(results):
        for name, t in zip(("out", "grad_value", "grad_sampling_loc", "grad_attn_weight"), tensors):
            n = t.numel()
            if n > sample:
                if n not in index:
                    g = torch.Generator().manual_seed(n)
                    index[n] = torch.randint(n, (sample,), generator=g).sort()[0].to(t.device)
                t = t.reshape(-1)[index[n]]
            np.save(os.path.join(path, f"layer{i}_{name}.npy"), t.detach().float().cpu().numpy())


def run_e2e(wl, layers, dev, dist_on, world, args):
    """Host buffers in, host buffers out, through MultiScaleDeformableAttnFunction.apply + backward.
    Three streams (H2D, compute, D2H) so that layer i+1's upload and layer i-1's download overlap layer
    i's kernels; device input buffers are double-buffered.  Every byte of value / locations / weights /
    grad_output goes host->device and every byte of output and the three gradients comes back, per layer."""
    import ir_ads_b200
    value, shapes, lsi, loc, w, go = layers[0]
    host_in = [t.cpu().pin_memory() for t in (value, loc, w, go)]
    out_shape = (wl.batch, wl.queries, wl.num_heads * wl.head_dim)
    host_out = [torch.empty(out_shape, dtype=value.dtype).pin_memory(), torch.empty_like(host_in[0]).pin_memory(),
                torch.empty_like(host_in[1]).pin_memory(), torch.empty_like(host_in[2]).pin_memory()]
    h2d = sum(t.numel() * t.element_size() for t in host_in)
    d2h = sum(t.numel() * t.element_size() for t in host_out)
    L = len(layers)
    steps = args.steps
    s_in, s_cmp, s_out = (torch.cuda.Stream(dev) for _ in range(3))
    dev_in = [[torch.empty_like(t, device=dev) for t in host_in] for _ in range(2)]
    ev = lambda: torch.cuda.Event()
    in_free = [ev(), ev()]      # compute finished reading dev_in[k]
    for e in in_free:
        e.record(s_cmp)

    def run(n_layers):
        for i in range(n_layers):
            k = i & 1
            with torch.cuda.stream(s_in):
                s_in.wait_event(in_free[k])
                for d, h in zip(dev_in[k], host_in):
                    d.copy_(h, non_blocking=True)
                ready = ev()
                ready.record(s_in)
            with torch.cuda.stream(s_cmp):
                s_cmp.wait_event(ready)
                v = dev_in[k][0].detach().requires_grad_(True)
                lo = dev_in[k][1].detach().requires_grad_(True)
                ww = dev_in[k][2].detach().requires_grad_(True)
                out = ir_ads_b200.MultiScaleDeformableAttnFunction.apply(v, shapes, lsi, lo, ww, 64)
                out.backward(dev_in[k][3])
                results = [out.detach(), v.grad, lo.grad, ww.grad]
                in_free[k] = ev()
                in_free[k].record(s_cmp)
                done = ev()
                done.record(s_cmp)
            with torch.cuda.stream(s_out):
                s_out.wait_event(done)
                for h, r in zip(host_out, results):
                    r.record_stream(s_out)
                    h.copy_(r, non_blocking=True)

    run(2)
    if dist_on:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(s_in)
    for _ in range(steps):
        run(L)
    t1.record(s_out)
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / steps
    if dist_on:
        from ir_ads_b200.sharding import max_over_ranks
        ms = max_over_ranks(ms, dev)
    return {"value": wl.points * L * world / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d * L,
            "d2h_bytes_per_step": d2h * L, "ms_per_step": ms, "steps": steps,
            "path": "pinned host -> H2D stream -> MultiScaleDeformableAttnFunction.apply + backward -> D2H stream "
                    "(out + 3 grads), 3-stream pipeline"}


def run_ref_cuda(layers, n_pts_layer):
    """The reference's own kernels (oracle/_ref, unmodified, sm_100a) on the same inputs and GPU."""
    try:
        from oracle import ref_cuda
        if not ref_cuda.available():
            return None
        bufs = None
        times_f, times_b = [], []
        for it in range(3):
            for value, shapes, lsi, loc, w, go in layers:
                if bufs is None:
                    bufs = (torch.empty_like(value), torch.empty_like(loc), torch.empty_like(w))
                    out = torch.empty_like(go)
                e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                e0.record()
                out.zero_()
                ref_cuda.forward(value, shapes, lsi, loc, w, out)
                e1.record()
                ref_cuda.backward(go, value, shapes, lsi, loc, w, bufs)
                e2.record()
                torch.cuda.synchronize()
                if it > 0:
                    times_f.append(e0.elapsed_time(e1))
                    times_b.append(e1.elapsed_time(e2))
        f, b = statistics.mean(times_f), statistics.mean(times_b)
        return {"value": n_pts_layer / ((f + b) * 1e-3), "unit": UNIT, "fwd_ms": f, "bwd_ms": b,
                "what": "reference ms_deformable_im2col/col2im kernels compiled for sm_100a, incl. its zero-fills"}
    except Exception as exc:  # a baseline must never take the bench down
        return {"error": repr(exc)}


if __name__ == "__main__":
    main()
