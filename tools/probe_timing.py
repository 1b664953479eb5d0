"""Card record and CUDA-event timing shared by the decode probes (region_probe, sample_probe, coarse_probe)."""
import subprocess

import numpy as np
import torch


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        info["power_limit_and_max_sm_clock"] = f"unavailable: {exc}"
    return info


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        ms.append(s.elapsed_time(e))
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    return out, {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "reps": reps,
                 "peak_torch_alloc_MB": peak / 2 ** 20}
