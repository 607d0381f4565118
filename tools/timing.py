"""What the timing scripts under tools/ share: the record of the card a number was measured on, the count of input
sets that keeps a timed call's reads out of L2, and the CUDA-event timing loop."""
import statistics
import subprocess

import torch

L2_BYTES = 126 * 2 ** 20   # the B200's L2


def rotations(set_bytes, lo, hi):
    """How many input sets of `set_bytes` to rotate over so that together they are three times the L2, clamped to
    [lo, hi]."""
    return max(lo, min(hi, -(-3 * L2_BYTES // set_bytes)))


def card():
    """{"device", "power_limit", "max_sm_clock"} of the card the numbers come from (the first one nvidia-smi lists).
    Raises without a CUDA device."""
    if not torch.cuda.is_available():
        raise RuntimeError("no CUDA device: the timing scripts measure on a GPU")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    _, power, clock = q.stdout.splitlines()[0].rsplit(",", 2)
    return {"device": torch.cuda.get_device_name(0), "power_limit": power.strip(), "max_sm_clock": clock.strip()}


def timed(arms, iters, warmup):
    """{name: [stages of one iteration, one tuple per rotating input set]} -> {name: [median ms of each stage]}.

    Every iteration runs each arm once, in dict order, on input set `iteration % len(sets)`, records a CUDA event
    before and after each stage and synchronises the device before the next arm starts.  The first `warmup`
    iterations are not counted."""
    times = {k: [] for k in arms}
    for it in range(warmup + iters):
        for name, per_set in arms.items():
            stages = per_set[it % len(per_set)]
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(stages) + 1)]
            ev[0].record()
            for i, stage in enumerate(stages):
                stage()
                ev[i + 1].record()
            torch.cuda.synchronize()
            if it >= warmup:
                times[name].append([ev[i].elapsed_time(ev[i + 1]) for i in range(len(stages))])
    return {k: [round(statistics.median(t[i] for t in v), 4) for i in range(len(v[0]))] for k, v in times.items()}
