"""Measurement helpers of the decoder and recogniser benchmarks (tools/bench_*decode.py, tools/bench_htr_train.py): the
card's name and power limit, CUDA-event timing, each kernel's device time from torch.profiler, and R's forward device time."""
import subprocess

import torch
from torch.profiler import ProfilerActivity, profile


def card():
    """The card's name, power limit and max SM clock from nvidia-smi (torch's device name without it)."""
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def timed_ms(fn, iters, warmup=5):
    """ms per call of fn from CUDA events around `iters` back-to-back calls after `warmup` calls (host launch overhead
    included when it exceeds the device time)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def kernel_us(fn, calls=20):
    """Device time per call of every kernel fn launches, {name: us}, from torch.profiler in a pass of its own after a warm-up
    call; memory copies and sets left out."""
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
        if t > 0 and not e.key.startswith(("Memcpy", "Memset")):
            out[e.key] = out.get(e.key, 0.0) + t / calls
    return out


def device_us(fn, names, calls=20):
    """Device time per call of the kernels whose name contains each of `names` (kernel_us): {name: us}."""
    per = kernel_us(fn, calls)
    return {n: sum(t for k, t in per.items() if n in k) for n in names}


def r_forward_us(R, rt, x, calls=10):
    """Device time of one forward pass of the recogniser R on x, all its kernels (kernel_us)."""
    return sum(kernel_us(lambda: R._logits(rt, x, False), calls).values())
