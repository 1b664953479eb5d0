#!/usr/bin/env python
"""Headline benchmark: NDMPS encode + truncate-to-chi + reconstruct voxels/s on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload cfg1|cfg2|cfg3|cfg4|cfg5b|cfg5] [--chi 64] [--dump-outputs DIR]

A step is one pass of the hot path over one BATCH of independent synthetic tensors (the reference's
benchmark loop walks a list of tensors, ``evaluation/benchmark.py:73-76,117-118``); ``--in-flight``
of them run concurrently per GPU (``imgcompressionmps.batch.VolumePipeline``: host threads x CUDA
streams).  Workloads (BASELINE.json configs, SURVEY section 8d):

  cfg3 (DEFAULT)  configs[2]: 512^3 fp32 volume, ``NDMPS.from_tensor(v, max_bond=64)`` + ``to_tensor`` -
                  the config the north-star target (>= 1 Gvoxel/s end to end on one B200) is quoted on.
                  With N > 1 ranks the same line also carries ``sharded``: ONE 512^3 volume column-sharded
                  over the N GPUs with an NCCL allreduce of the bond-sized Gram matrix per sweep step.
  cfg2            configs[1]: 256^3 volume, chi sweep 128/64/32/16/8 with fidelity vs the chi = 128 state,
                  3-D SSIM and PSNR inside the step (voxels are counted once per chi).
  cfg1            configs[0]: 256 x 256 image at chi = 32 + PSNR + SSIM.
  cfg4            configs[3]: fMRI subjects (64, 64, 32, 400) at chi = 64 + 4-D SSIM, subjects sharded one per slot.
  cfg5b           configs[4], partition 5-B: (1920, 1080, 64) channel chunks, DCT mode, chi = 64.
  cfg5            the literal configs[4] shape (1920, 1080, 3, 512): degenerate (one site), reported as such.

* ``value``  : device-resident - the tensors already sit in HBM, the results stay in HBM.  K steps timed
  with CUDA events, barrier + synchronize on both sides, max over ranks.  When the distinct inputs of a
  step are several times the L2 (cfg3: 1.07 GB) the K steps run back to back inside one event pair - the
  queue keeps ``in_flight`` tensors in flight across step boundaries; otherwise, and with ``--per-step``,
  each step has its own event pair and the L2 is flushed between steps (outside the pairs).  ``run`` says which.
* ``e2e``    : the same K steps from pinned HOST buffers (H2D copy of every input and D2H copy of every
  reconstruction inside the timed region; cfg3 goes through the C ABI entry ``ndmps_roundtrip_host``),
  host clock around the K steps with a synchronize on both sides.
* ``single`` : one tensor at a time (latency) with the library's stage profiler on; the rooflines come
  from this pass and the top-level ``roofline`` is the stage with the largest share of it.
* ``--impl reference``: the CPU oracle (numpy/LAPACK float64 restatement of the reference path - the
  reference itself cannot be imported without quimb / scikit-image) on the SAME workload, one tensor
  per step, all host threads, rank 0 only; the number of steps is bounded by ``--ref-budget`` seconds.
* ``--dump-outputs DIR``: what the device-resident path computed in its last timed step, as .npy files (see
  ``write_outputs``).  Inputs are seeded, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import csv
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
for _p in (str(ROOT), str(ROOT / "img-compression-mps_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "ndmps_encode_truncate_reconstruct_voxels_per_s"
UNIT = "voxels/s"
L2_BYTES = 126 << 20          # B200 L2: timed iterations either flush it or work on inputs several times larger
DUMP_LIMIT = 64 << 20         # --dump-outputs writes at most this many bytes
DUMP_SEED = 0

CHI_SWEEP = (128, 64, 32, 16, 8)
WORKLOADS = {
    "cfg1": {"shape": (256, 256), "chi": 32, "mode": "Std", "in_flight": 8, "batch": 64, "passes": 1,
             "name": "configs[0]: 256x256 fp32 synthetic image, chi = 32, reconstruct + PSNR + SSIM"},
    "cfg2": {"shape": (256, 256, 256), "chi": 128, "mode": "Std", "in_flight": 8, "batch": 16, "passes": len(CHI_SWEEP),
             "name": "configs[1]: 256x256x256 fp32 synthetic MRI volume, chi sweep 128/64/32/16/8 + fidelity + 3-D SSIM + PSNR"},
    "cfg3": {"shape": (512, 512, 512), "chi": 64, "mode": "Std", "in_flight": 8, "batch": 16, "passes": 1,
             "name": "configs[2]: 512x512x512 fp32 synthetic volume, chi = 64, encode + TT-SVD + reconstruct (north-star target)"},
    "cfg4": {"shape": (64, 64, 32, 400), "chi": 64, "mode": "Std", "in_flight": 4, "batch": 8, "passes": 1,
             "name": "configs[3]: 64x64x32x400 fp32 synthetic fMRI subjects, chi = 64, reconstruct + 4-D SSIM"},
    "cfg5b": {"shape": (1920, 1080, 64), "chi": 64, "mode": "DCT", "in_flight": 3, "batch": 3, "passes": 1,
              "name": "configs[4] partition 5-B: 1920x1080x64 fp32 video channel chunks, DCT mode, chi = 64"},
    "cfg5": {"shape": (1920, 1080, 3, 512), "chi": 64, "mode": "DCT", "in_flight": 1, "batch": 1, "passes": 1,
             "name": "configs[4] literal shape 1920x1080x3x512: degenerate under the reference's encoding (one site)"},
}


def synthetic_volume(shape, seed):
    """Ellipsoid phantom + smooth texture + 0.02 noise inside the object, exact-zero background
    (SURVEY section 8d).  Built per z-slab to keep host memory flat."""
    rng = np.random.default_rng(seed)
    params = [(rng.uniform(-0.25, 0.25, 3), rng.uniform(0.35, 0.8, 3) * (1.0 - 0.18 * k), 0.25 + 0.1 * k) for k in range(4)]
    axes = [np.linspace(-1, 1, n, dtype=np.float32) for n in shape]
    out = np.empty(shape, dtype=np.float32)
    gy, gz = np.meshgrid(axes[1], axes[2], indexing="ij")
    for i, xv in enumerate(axes[0]):
        sl = np.zeros(shape[1:], dtype=np.float32)
        for c, r, amp in params:
            r2 = ((xv - c[0]) / r[0]) ** 2 + ((gy - c[1]) / r[1]) ** 2 + ((gz - c[2]) / r[2]) ** 2
            sl += amp / (1.0 + np.exp(np.clip((r2 - 1.0) * 12.0, -60, 60)))
        inside = sl > 0.05
        sl += 0.05 * np.cos(3 * xv) * np.cos(3 * gy + 1) * np.cos(3 * gz + 2) * inside
        sl += 0.02 * rng.random(shape[1:], dtype=np.float32) * inside
        sl[sl < 0.02] = 0.0
        out[i] = sl
    return out


def synthetic_image(shape=(256, 256), seed=2025):
    """configs[0]: smooth + texture grayscale image, clip(sum of 3 Gaussians + 0.05 noise, 0, 1) (SURVEY 8d)."""
    rng = np.random.default_rng(seed)
    gy, gx = np.meshgrid(np.linspace(-1, 1, shape[0]), np.linspace(-1, 1, shape[1]), indexing="ij")
    img = np.zeros(shape)
    for _ in range(3):
        cy, cx = rng.uniform(-0.5, 0.5, 2)
        sy, sx = rng.uniform(0.15, 0.5, 2)
        img += rng.uniform(0.3, 0.6) * np.exp(-(((gy - cy) / sy) ** 2 + ((gx - cx) / sx) ** 2))
    img += 0.05 * rng.random(shape)
    return np.clip(img, 0.0, 1.0).astype(np.float32)


def synthetic_fmri(shape=(64, 64, 32, 400), seed=3000):
    """configs[3]: static phantom x (1 + 0.05 low-rank temporal modes (rank 8, sinusoids)) + 0.01 noise (SURVEY 8d)."""
    rng = np.random.default_rng(seed)
    sx, sy, sz, nt = shape
    g = np.meshgrid(*[np.linspace(-1, 1, n, dtype=np.float32) for n in (sx, sy, sz)], indexing="ij")
    base = np.zeros((sx, sy, sz), dtype=np.float32)
    for k in range(3):
        c = rng.uniform(-0.2, 0.2, 3)
        r = rng.uniform(0.45, 0.85, 3) * (1.0 - 0.2 * k)
        r2 = sum(((gi - ci) / ri) ** 2 for gi, ci, ri in zip(g, c, r))
        base += (0.3 + 0.15 * k) / (1.0 + np.exp(np.clip((r2 - 1.0) * 10.0, -60, 60)))
    t = np.arange(nt, dtype=np.float32) / nt
    out = np.empty(shape, dtype=np.float32)
    mod = np.ones(shape, dtype=np.float32)
    for m in range(8):
        spatial = np.cos((m % 3 + 1) * g[0] + m) * np.cos((m % 2 + 1) * g[1] - m) * np.cos((m % 4) * 0.5 * g[2])
        temporal = np.sin(2 * np.pi * (m + 1) * t + rng.uniform(0, 6.28))
        mod += (0.05 / (1 + 0.5 * m)) * spatial[..., None].astype(np.float32) * temporal[None, None, None, :].astype(np.float32)
    np.multiply(base[..., None], mod, out=out)
    out += 0.01 * rng.random(shape, dtype=np.float32)
    return out


def synthetic_video(shape=(1920, 1080, 64), seed=4000, channel=0, chunk=0):
    """configs[4], non-degenerate partition 5-B (SURVEY 8d): one colour channel x one 64-frame chunk of a moving-blob
    video: 5 Gaussians with linear motion, per-channel gain, 0.02 noise."""
    rng = np.random.default_rng(seed)
    blobs = [(rng.uniform(-0.6, 0.6, 2), rng.uniform(-0.4, 0.4, 2), rng.uniform(0.1, 0.35, 2), rng.uniform(0.3, 0.8)) for _ in range(5)]
    gains = rng.uniform(0.6, 1.0, 3)
    noise = np.random.default_rng(seed + 17 * channel + 101 * chunk + 1)
    w, h, nf = shape
    gx = np.linspace(-1, 1, w, dtype=np.float32)[:, None]
    gy = np.linspace(-1, 1, h, dtype=np.float32)[None, :]
    out = np.empty(shape, dtype=np.float32)
    for f in range(nf):
        tt = (chunk * nf + f) / 512.0
        fr = np.zeros((w, h), dtype=np.float32)
        for p0, vel, sig, amp in blobs:
            cx, cy = p0[0] + vel[0] * tt, p0[1] + vel[1] * tt
            fr += np.float32(amp) * (np.exp(-((gx - np.float32(cx)) / np.float32(sig[0])) ** 2) * np.exp(-((gy - np.float32(cy)) / np.float32(sig[1])) ** 2))
        fr *= np.float32(gains[channel])
        fr += 0.02 * noise.random((w, h), dtype=np.float32)
        out[:, :, f] = fr
    return out


def algorithmic_work(dims, ranks):
    """Bytes / flops of the stages per SURVEY section 8(d) for float32 payloads (4 B)."""
    L, n = len(dims), int(np.prod(dims))
    r = [1] + list(ranks) + [1]
    sweep_bytes = gram_flops = proj_flops = proj_bytes = 0.0
    cols = n
    for i in range(L - 1):
        m = r[i] * dims[i]
        cols //= dims[i]
        sweep_bytes += 4.0 * (2 * m * cols + r[i + 1] * cols)
        proj_bytes += 4.0 * (m * cols + r[i + 1] * cols)
        gram_flops += 2.0 * m * m * cols
        proj_flops += 2.0 * m * r[i + 1] * cols
    recon_bytes = recon_flops = 0.0
    p = 1
    for k in range(L):
        recon_bytes += 4.0 * (p * r[k] + p * dims[k] * r[k + 1])
        recon_flops += 2.0 * p * r[k] * dims[k] * r[k + 1]
        p *= dims[k]
    # Gram passes actually executed: sites are front-merged while the fused row count stays <= 512
    executed = issued = issued_i8 = i8_time_share = proj_bytes_exec = gram_bytes_exec = 0.0
    cols, i, rprev = n, 0, 1
    while i < L - 1:
        rows = rprev * dims[i]
        cols //= dims[i]
        k = 1
        while i + k < L - 1 and rows * dims[i + k] <= 512 and rows * dims[i + k] <= cols // dims[i + k]:
            rows *= dims[i + k]
            cols //= dims[i + k]
            k += 1
        side = min(rows, cols)
        executed += 2.0 * side * side * max(rows, cols)
        nt = -(-side // 128)                                  # gram_dmma computes the upper-triangle 128 x 128 tiles only
        issued += 2.0 * side * side * max(rows, cols) * ((nt + 1) / (2.0 * nt) if side >= 48 else 1.0)
        # tc_gemm.cu gram_tc: float32 unfoldings with 64 <= rows <= 4096 and >= 2048 columns go through the integer
        # tensor cores: 128 x 64 tiles that touch the upper triangle, 15 digit products (kind::i8) per 32-deep k-step
        if rows <= cols and 64 <= rows <= 4096 and cols >= 2048:
            ntr, ntc = -(-rows // 128), -(-rows // 64)
            tiles = sum(max(ntc - 2 * ti, 0) for ti in range(ntr))
            issued_i8 += 15.0 * 2.0 * tiles * 128 * 64 * cols
        gram_bytes_exec += 4.0 * rows * cols
        proj_bytes_exec += 4.0 * (rows * cols + r[i + k] * cols)
        rprev = r[i + k]
        i += k
    return {"encode_bytes": 8.0 * n, "decode_bytes": 8.0 * n, "sweep_bytes": sweep_bytes, "gram_flops": gram_flops,
            "gram_flops_executed": executed, "gram_flops_issued": issued, "gram_bytes_executed": gram_bytes_exec,
            "project_bytes_executed": proj_bytes_exec, "gram_i8_ops_issued": issued_i8,
            "recon_bytes_executed": 4.0 * n + 4.0 * (int(np.prod(dims[: (L + 1) // 2])) + int(np.prod(dims[(L + 1) // 2:]))) * max(ranks),
            "project_flops": proj_flops, "project_bytes": proj_bytes, "recon_bytes": recon_bytes, "recon_flops": recon_flops}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, enabled=True):
        self.index, self.rows, self.proc, self.enabled = index, [], None, enabled

    def __enter__(self):
        if not self.enabled:                 # NVML queries take driver-wide locks: one sampler per node, not one per rank
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, val in zip(names, r[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def _all_host_threads():
    """Context manager giving BLAS every host core (torchrun exports OMP_NUM_THREADS=1)."""
    try:
        from threadpoolctl import threadpool_limits
        return threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        import contextlib
        return contextlib.nullcontext()


def _all_host_threads():
    """Context manager giving BLAS every host core (torchrun exports OMP_NUM_THREADS=1)."""
    try:
        from threadpoolctl import threadpool_limits
        return threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        import contextlib
        return contextlib.nullcontext()


def host_threads():
    try:
        from threadpoolctl import threadpool_info
        with _all_host_threads():
            n = max((p.get("num_threads", 1) for p in threadpool_info()), default=1)
        return int(n)
    except Exception:
        return os.cpu_count() or 1


# ---------------------------------------------------------------------------------------------
# the workloads: inputs, the per-tensor unit of work on the device, the same unit on the CPU oracle
# ---------------------------------------------------------------------------------------------
def make_input(workload, rank, i):
    shape = WORKLOADS[workload]["shape"]
    if workload == "cfg1":
        return synthetic_image(shape, 2025 + 64 * rank + i)
    if workload == "cfg2":
        return synthetic_volume(shape, 2026 + 16 * rank + i)
    if workload == "cfg3":
        return synthetic_volume(shape, 2027 + 16 * rank + i)
    if workload == "cfg4":
        return synthetic_fmri(shape, 3000 + 64 * rank + i)
    if workload == "cfg5b":
        j = 3 * rank + i
        return synthetic_video(shape, 4000, channel=j % 3, chunk=(j // 3) % 8)
    raise ValueError(workload)


def workload_config(workload, args, world):
    """The `config` object of the JSON line: a function of the command line only, identical for both arms."""
    wl = WORKLOADS[workload]
    chis = list(CHI_SWEEP) if workload == "cfg2" else [wl["chi"] if args.chi == 0 else args.chi]
    return {"workload": wl["name"], "key": workload, "shape": list(wl["shape"]), "chi": chis, "mode": wl["mode"],
            "dtype_in": "float32", "voxel_passes_per_tensor": wl["passes"],
            "unit": "per tensor: NDMPS.from_tensor(x, mode, max_bond=chi) + to_tensor" +
                    {"cfg1": " + compute_psnr + compute_ssim_2d", "cfg2": " per chi + compute_overlap vs chi=128 + avg_ssim_3d + compute_psnr",
                     "cfg4": " + avg_ssim_4d"}.get(workload, "")}


def device_unit(workload, chi):
    """f(volume on device) -> (reconstruction to hand back or None, dict of scalars)."""
    from imgcompressionmps.core.ndmps import NDMPS
    from imgcompressionmps.utils.metrics import compute_overlap, compute_psnr, compute_ssim_by_dim
    mode = WORKLOADS[workload]["mode"]

    def plain(v):
        obj = NDMPS.from_tensor(v, mode=mode, max_bond=chi)
        return obj.to_tensor_device(), {"bond_dims": obj.bond_sizes(), "site_dims": obj.mps.site_dims}

    def with_metrics(v):
        obj = NDMPS.from_tensor(v, mode=mode, max_bond=chi)
        rec = obj.to_tensor_device()
        out = {"bond_dims": obj.bond_sizes(), "site_dims": obj.mps.site_dims, "ssim": compute_ssim_by_dim(rec, v)}
        if workload == "cfg1":
            out["psnr"] = compute_psnr(rec, v)
        return None, out

    def chi_sweep(v):
        ref = NDMPS.from_tensor(v, max_bond=CHI_SWEEP[0])
        out = {"site_dims": ref.mps.site_dims, "bond_dims": {}, "fidelity": {}, "ssim": {}, "psnr": {}}
        for c in CHI_SWEEP:
            obj = ref if c == CHI_SWEEP[0] else NDMPS.from_tensor(v, max_bond=c)
            rec = obj.to_tensor_device()
            out["bond_dims"][c] = obj.bond_sizes()
            out["fidelity"][c] = compute_overlap(obj, ref)
            out["ssim"][c] = compute_ssim_by_dim(rec, v)
            out["psnr"][c] = compute_psnr(rec, v)
        return None, out

    return {"cfg1": with_metrics, "cfg2": chi_sweep, "cfg3": plain, "cfg4": with_metrics, "cfg5b": plain}[workload]


def dump_positions(nvox, batch):
    """Flat voxel positions of each reconstruction that --dump-outputs keeps: all of them when a step's tensors fit in
    3/4 of DUMP_LIMIT (counted as float64), otherwise the same subset for every tensor: one position drawn from
    numpy's default_rng(DUMP_SEED) in each of `keep` equal strata of the flat index, so two runs or two builds keep
    the same voxels, spread over the whole tensor, without materialising a permutation of all of them."""
    keep = max(1, (DUMP_LIMIT * 3 // 4) // (8 * batch))
    if keep >= nvox:
        return np.arange(nvox)
    edges = np.arange(keep + 1, dtype=np.int64) * nvox // keep
    return edges[:-1] + (np.random.default_rng(DUMP_SEED).random(keep) * np.diff(edges)).astype(np.int64)


def write_outputs(out_dir, results):
    """--dump-outputs: ``results`` holds, for each tensor of the last timed step, (its kept reconstruction voxels or
    None, the unit's scalars).  One DIR/<name>.npy per name with the step's tensors along axis 0: ``reconstruction``
    (float32), then every scalar and bond list of the unit as float64 (``<name>_chi<c>`` for the chi sweep's entries)."""
    arrays = {}
    if results[0][0] is not None:
        arrays["reconstruction"] = np.stack([r.cpu().numpy() for r, _ in results])
    for key, first in results[0][1].items():
        for sub in (list(first) if isinstance(first, dict) else [None]):
            vals = [s[key] if sub is None else s[key][sub] for _, s in results]
            arrays[key if sub is None else f"{key}_chi{sub}"] = np.asarray(vals, dtype=np.float64)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT}-byte limit (fewer --volumes)")
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", a)


def oracle_unit(workload, chi):
    """The same unit of work on the CPU oracle (numpy / LAPACK float64, oracle/)."""
    from oracle import metrics as OM
    from oracle.ndmps import OracleNDMPS
    mode = WORKLOADS[workload]["mode"]

    def plain(x):
        OracleNDMPS.from_tensor(x, mode=mode, max_bond=chi).to_tensor()

    def with_metrics(x):
        x64 = x.astype(np.float64)
        rec = OracleNDMPS.from_tensor(x, mode=mode, max_bond=chi).to_tensor()
        OM.compute_ssim_by_dim(rec, x64)
        if workload == "cfg1":
            OM.compute_psnr(rec, x64)

    def chi_sweep(x):
        x64 = x.astype(np.float64)
        ref = OracleNDMPS.from_tensor(x, max_bond=CHI_SWEEP[0])
        for c in CHI_SWEEP:
            obj = ref if c == CHI_SWEEP[0] else OracleNDMPS.from_tensor(x, max_bond=c)
            rec = obj.to_tensor()
            OM.compute_overlap(obj.cores, obj.norm_value, ref.cores, ref.norm_value)
            OM.compute_ssim_by_dim(rec, x64)
            OM.compute_psnr(rec, x64)

    return {"cfg1": with_metrics, "cfg2": chi_sweep, "cfg3": plain, "cfg4": with_metrics, "cfg5b": plain}[workload]


def degenerate_report(args):
    """configs[4] as literally written: (1920, 1080, 3, 512).  The size-3 axis has one prime factor, so the
    reference's get_factorlist balances every axis to ONE level: a single-site MPS of dimension 3 185 049 600,
    nothing to truncate, compress() loops over range(1, 1) (SURVEY section 0.5).  Reported, not replaced silently;
    the non-degenerate partition of the same data is workload cfg5b."""
    from imgcompressionmps.utils.core import get_factorlist
    shape = WORKLOADS["cfg5"]["shape"]
    factors, _ = get_factorlist(shape)
    line = {"metric": METRIC, "value": None, "unit": UNIT, "n_gpus": args.gpus, "steps": 0, "warmup": 0, "ms_per_step": None,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOADS["cfg5"]["name"], "key": "cfg5", "shape": list(shape)},
            "degenerate": {"levels": int(factors.shape[0]), "site_dims": [int(np.prod(f)) for f in factors],
                           "bonds": [], "note": "L = 1: from_tensor stores the permuted tensor as one core, compress() is a no-op, "
                                                "to_tensor is the inverse permutation; there is no chi to hold fixed. "
                                                "Use --workload cfg5b (3 channels x 8 chunks of 64 frames)."}}
    # the one-site path itself, on a reduced-frame tensor of the same axis structure
    try:
        import torch
        if torch.cuda.is_available():
            from imgcompressionmps.core.ndmps import NDMPS
            small = np.random.default_rng(0).random((192, 108, 3, 8)).astype(np.float32)
            obj = NDMPS.from_tensor(small, mode="DCT", max_bond=args.chi or 64)
            obj.compress(0.1)
            line["degenerate"]["one_site_path_check"] = {"shape": list(small.shape), "bonds": obj.bond_sizes(),
                                                         "roundtrip_max_abs_err": float(np.abs(obj.to_tensor() - small).max())}
    except Exception as exc:   # the report itself needs no GPU
        line["degenerate"]["one_site_path_check"] = f"skipped: {exc}"
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# --impl reference : the CPU oracle on the same workload
# ---------------------------------------------------------------------------------------------
def time_oracle(workload, chi, x, max_steps, budget_s):
    """(voxels/s, seconds per tensor, steps run): at least one step, more while the budget lasts."""
    unit = oracle_unit(workload, chi)
    passes = WORKLOADS[workload]["passes"]
    times = []
    with _all_host_threads():
        t_all = time.perf_counter()
        while len(times) < max_steps:
            t0 = time.perf_counter()
            unit(x)
            times.append(time.perf_counter() - t0)
            if time.perf_counter() - t_all + times[-1] > budget_s:
                break
    per = float(np.mean(times))
    return x.size * passes / per, per, len(times)


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    workload = args.workload
    wl = WORKLOADS[workload]
    chi = args.chi or wl["chi"]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    x = make_input(workload, 0, 0)
    warm = 0
    with _all_host_threads():                                  # spin the BLAS pool up on a small tensor of the family
        from oracle.ndmps import OracleNDMPS
        OracleNDMPS.from_tensor(np.random.default_rng(0).random((32, 32, 32)).astype(np.float32), max_bond=8).to_tensor()
    if workload in ("cfg1",):                                  # cheap enough for real warm-up steps
        warm = args.warmup
        for _ in range(warm):
            oracle_unit(workload, chi)(x)
    value, per, steps = time_oracle(workload, chi, x, args.steps, args.ref_budget)
    cores = host_threads()
    sample = (f"one tensor of the workload per step ({'x'.join(map(str, wl['shape']))} float32, the first tensor of rank 0's batch), "
              f"{steps} of the {args.steps} requested steps run within the {args.ref_budget:.0f} s budget, "
              f"{warm} warm-up steps (a 32^3 run spins the BLAS threads up); numpy/LAPACK float64, {cores} threads")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": 1e3 * per, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(workload, args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "steps_requested": args.steps, "warmup_requested": args.warmup,
        "note": "reference cannot be imported (quimb, scikit-image absent): oracle port timed on host cores, same workload "
                "and shape as the GPU arm; fewer steps than requested when one tensor takes tens of seconds",
    }))


# ---------------------------------------------------------------------------------------------
# rooflines
# ---------------------------------------------------------------------------------------------
def load_peaks():
    peaks = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback"}
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        m = json.loads(pk.read_text())
        peaks = {"hbm_gbs": m["hbm_gbs"], "bf16_tflops": m.get("bf16_tflops_sustained", m["bf16_tflops"]),
                 "bf16_tflops_burst": m["bf16_tflops"], "source": "measured"}
    return peaks


def measure_fp64_rate(torch):
    """FP64 FMA rate of this GPU, measured in the run (cuBLAS DGEMM 4096^3 through torch, best of 5): the
    denominator of the latency-bound float64 stages.  torch is the yardstick here, not the product."""
    a = torch.rand((4096, 4096), dtype=torch.float64, device="cuda")
    b = torch.rand((4096, 4096), dtype=torch.float64, device="cuda")
    best = None
    for _ in range(6):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        torch.matmul(a, b)
        e.record()
        e.synchronize()
        ms = s.elapsed_time(e)
        best = ms if best is None else min(best, ms)
    return 2.0 * 4096 ** 3 / (best * 1e-3) / 1e12


def ncu_traffic(kernel_substring):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of a kernel, from the newest
    ``ncu --set full`` raw-page CSV committed under profiles/ (None when no capture names the kernel)."""
    best = None
    for path in sorted((ROOT / "profiles").glob("r*_kernels_raw.csv"), reverse=True):
        try:
            rows = list(csv.reader(open(path, newline="")))
            hdr, units = rows[0], rows[1]
            ik, ir, iw = hdr.index("Kernel Name"), hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            for r in rows[2:]:
                if kernel_substring in r[ik]:
                    val = float(r[ir]) * scale.get(units[ir], 1.0) + float(r[iw]) * scale.get(units[iw], 1.0)
                    best = {"bytes": val, "source": f"profiles/{path.name}", "kernel": r[ik][:80]} if best is None or val > best["bytes"] else best
            if best:
                return best
        except Exception:
            continue
    return None


def build_rooflines(stages_per_call, single_ms, work, nvox, peaks, fp64_tflops, eig_flops, used_tc, bit_permute=False):
    """stage -> roofline entry.  stages_per_call: {stage: (ms per tensor, calls per tensor)}."""
    out = {}

    def entry(stage, kernel, bound, achieved, peak, unit, traffic_key, extra=None):
        ms, calls = stages_per_call[stage]
        e = {"stage": stage, "kernel": kernel, "bound": bound, "achieved": achieved, "peak": peak, "unit": unit,
             "frac": achieved / peak if peak else None, "ms_per_tensor": ms, "calls_per_tensor": calls,
             "share_of_tensor_time": ms / single_ms if single_ms else None}
        t = ncu_traffic(traffic_key) if traffic_key else None
        e["traffic"] = t["bytes"] if t else None
        if t:
            e["traffic_source"] = t["source"]
        if extra:
            e.update(extra)
        out[stage] = e

    def have(stage):
        return stage in stages_per_call and stages_per_call[stage][1] > 0 and stages_per_call[stage][0] > 0

    if have("permute"):
        ms = stages_per_call["permute"][0]
        b = work["encode_bytes"] + work["decode_bytes"]
        name = ("permute_bits_kernel (power-of-two shape: register bit-permutation, two 16-byte loads + two 16-byte stores per "
                "thread, no shared memory; encode + decode)") if bit_permute else "permute_tiled_kernel<float,4> (encode + decode)"
        entry("permute", name, "hbm", b / (ms * 1e-3) / 1e9, peaks["hbm_gbs"], "GB/s",
              "permute_bits_kernel" if bit_permute else "permute_tiled_kernel", {"algorithmic_bytes_per_tensor": b})
    if have("gram"):
        ms = stages_per_call["gram"][0]
        f = work["gram_flops_executed"]
        if used_tc and work.get("gram_i8_ops_issued"):
            ops = work["gram_i8_ops_issued"]
            entry("gram", "gram_i8_kernel (tcgen05.mma kind::i8 on five 7-bit digit planes: 15 digit products per k-step issued as 6 "
                          "stacked-plane MMAs, int32 TMEM accumulators, float64 drain) + row_stats / split_i8 passes; small "
                          "unfoldings on the FP64 tensor pipe",
                  "tensor", ops / (ms * 1e-3) / 1e12, 2.0 * peaks["bf16_tflops"], "TOP/s (int8)", "gram_i8_kernel",
                  {"algorithmic_fp32_flops_per_tensor": f, "issued_int8_ops_per_tensor": ops,
                   "peak_note": "2 x the measured dense bf16 rate of MEASURED_PEAKS.json (kind::i8 issues at twice the kind::f16 rate; "
                                "no measured int8 figure exists for this pool)",
                   "note": "achieved = int8 tensor-core operations issued by gram_i8_kernel (tiles touching the upper triangle) / time of "
                           "the whole Gram stage, which also holds the statistics and digit-split passes (HBM-bound) and the small "
                           "Grams; profiles/r02_summary.md has the kernel alone (tensor pipe 77 % active under ncu)"})
        else:
            entry("gram", "gram_dmma_kernel (FP64 tensor pipe, mma.sync m8n8k4.f64)", "tensor", f * work["gram_upper_fraction"] / (ms * 1e-3) / 1e12,
                  fp64_tflops, "TFLOP/s (fp64)", "gram_dmma_kernel", {"algorithmic_fp32_flops_per_tensor": f})
    if have("project"):
        ms = stages_per_call["project"][0]
        b = work["project_bytes_executed"]
        entry("project", "projection T = P^T M (one pass per front-merged group; proj_i8_kernel on the Gram's int8 digit planes)" if used_tc
              else "projection T = P^T M (one pass per front-merged group)", "hbm", b / (ms * 1e-3) / 1e9, peaks["hbm_gbs"], "GB/s",
              "proj_i8_kernel" if used_tc else "gemm_dmma_kernel", {"algorithmic_bytes_per_tensor": b, "survey_bytes_per_tensor_one_pass_per_site": work["project_bytes"],
               "flops_per_tensor": work["project_flops"]})
    if have("contract"):
        ms = stages_per_call["contract"][0]
        b = work["recon_bytes_executed"]
        entry("contract", "core chain (bond-sized) + final product dense = X W (gemm_tc_kernel, bf16x3 on tcgen05)", "hbm",
              b / (ms * 1e-3) / 1e9, peaks["hbm_gbs"], "GB/s", "gemm_tc_kernel" if used_tc else "gemm_dmma_kernel",
              {"algorithmic_bytes_per_tensor": b, "survey_bytes_per_tensor_site_by_site": work["recon_bytes"],
               "flops_per_tensor": work["recon_flops"],
               "note": "bytes = what this implementation has to move: the dense tensor written once plus the two half-chain factors "
                       "(SURVEY 8(d) counts a site-by-site chain that re-reads the growing intermediate: kept for reference)"})
    if have("eig"):
        ms = stages_per_call["eig"][0]
        entry("eig", "bond eigenproblems: eig_topk.cu (tridiag_kernel, bisect, invit, Rayleigh-Ritz) for capped bonds, eig.cu Jacobi otherwise",
              "tensor", eig_flops / (ms * 1e-3) / 1e12, fp64_tflops, "TFLOP/s (fp64)", "tridiag_kernel",
              {"flops_per_tensor": eig_flops, "peak_source": "cuBLAS DGEMM 4096^3 timed in this run (FP64 tensor pipe)",
               "bound_note": "latency-bound in fact: float64 SIMT work in chains of dependent steps (n - 2 Householder columns of ~2.6 us "
                             "per 512 x 512 bond matrix, each two block reductions + a cluster-wide exchange); neither HBM traffic (2 MB per "
                             "solve) nor a tensor pipe limits it.  The FP64 rate is the only roofline its flops can be put against, "
                             "so `frac` says how far a dependency chain is from a throughput bound, not how well a pipe is fed"})
    if have("metric"):
        ms = stages_per_call["metric"][0]
        b = work.get("metric_bytes", 0.0)
        if b:
            entry("metric", "ssim.cu (per-slice range + 7x7 box moments) / psnr reduction", "hbm", b / (ms * 1e-3) / 1e9, peaks["hbm_gbs"], "GB/s",
                  "ssim_", {"algorithmic_bytes_per_tensor": b})
    if have("dct"):
        ms = stages_per_call["dct"][0]
        b = 16.0 * nvox
        entry("dct", "last-axis DCT-II + DCT-III (cosine matrix GEMM)", "hbm", b / (ms * 1e-3) / 1e9, peaks["hbm_gbs"], "GB/s", "dct", {"algorithmic_bytes_per_tensor": b})
    return out


def work_for(workload, info, nvox):
    """Algorithmic bytes / flops of ONE tensor of the workload (SURVEY 8d), summed over the chi sweep for cfg2."""
    dims = info["site_dims"]
    bonds = info["bond_dims"]
    per_chi = [bonds[c] for c in CHI_SWEEP] if isinstance(bonds, dict) else [bonds]
    tot = None
    for ranks in per_chi:
        w = algorithmic_work(dims, ranks)
        tot = w if tot is None else {k: tot[k] + w[k] for k in w}
    n = len(per_chi)
    tot["gram_upper_fraction"] = tot["gram_flops_issued"] / tot["gram_flops_executed"] if tot["gram_flops_executed"] else 1.0
    ndim = len(WORKLOADS[workload]["shape"])
    if workload in ("cfg1", "cfg2", "cfg4"):          # SSIM 16 B/voxel (+ PSNR 8 B/voxel where it is computed)
        tot["metric_bytes"] = n * nvox * 4.0 * (4 + (2 if workload in ("cfg1", "cfg2") else 0)) * (1 if ndim else 1)
    return tot


# ---------------------------------------------------------------------------------------------
# ours
# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    from imgcompressionmps import _native, _ops
    from imgcompressionmps.batch import VolumePipeline

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU path for --impl ours")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # NCCL's banner / debug lines stay off stdout (one JSON line)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    workload = args.workload
    wl = WORKLOADS[workload]
    chi = args.chi or wl["chi"]
    shape = wl["shape"]
    nvox = int(np.prod(shape))
    passes = wl["passes"]
    in_flight = args.in_flight or wl["in_flight"]
    batch = args.volumes or wl["batch"]
    n_distinct = min(batch, 2 if nvox > (1 << 26) else 4)              # distinct inputs; L2 is flushed between steps
    hosts = [make_input(workload, rank, i) for i in range(n_distinct)]
    pinned = [torch.from_numpy(h).pin_memory() for h in hosts]
    vols_distinct = [p.cuda(non_blocking=False) for p in pinned]
    vols = [vols_distinct[i % n_distinct] for i in range(batch)]
    ctx = _native.context()
    flush_buf = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device="cuda")   # > 126 MB L2
    pipe = VolumePipeline(workers=in_flight)
    unit = device_unit(workload, chi)
    keep = torch.from_numpy(dump_positions(nvox, batch)).cuda() if args.dump_outputs else None

    def timed(item):
        if isinstance(item, tuple):  # last step with --dump-outputs: the unit + one gather of the kept voxels
            rec, scal = unit(item[0])
            return (None if rec is None else rec.reshape(-1).index_select(0, keep)), scal
        return unit(item)[1]

    def step_items(last_step):
        return [(v,) for v in vols] if last_step and keep is not None else vols

    def step(last_step=False):
        return pipe.map(timed, step_items(last_step))

    info = None
    for _ in range(max(args.warmup, 3)):
        rec, info = unit(vols[0])
        step()
    torch.cuda.synchronize()
    err = None
    if rec is not None:
        err = float(torch.linalg.vector_norm((rec - vols[0]).double()) / torch.linalg.vector_norm(vols[0].double()))
    del rec

    # ---- device-resident timing: `batch` tensors per step, `in_flight` of them concurrently ---------------
    # The K steps run back to back inside ONE event pair (barrier + synchronize on both sides) when the distinct inputs
    # of a step are several times the 126 MB L2 - nothing a step reads can still be cached from the one before, so no flush
    # is needed and the pipeline keeps `in_flight` tensors in flight across step boundaries, as a production queue would.
    # Otherwise (and with --per-step) every step has its own event pair and the L2 is flushed between steps.
    back_to_back = (not args.per_step) and n_distinct * nvox * 4 >= 4 * L2_BYTES
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    launches0 = pipe.launch_count()
    barrier()
    with ClockSampler(local, enabled=(rank == 0)) as clocks:
        if back_to_back:
            flush_buf.fill_(0)
            starts[0].record()
            last = pipe.map(timed, vols * (args.steps - 1) + step_items(True))[-batch:]
            stops[0].record()
        else:
            for i in range(args.steps):
                flush_buf.fill_(i & 0xFF)                            # evict L2 (outside the event pair)
                starts[i].record()
                last = step(i == args.steps - 1)                     # workers wait for the submitting stream, then are joined
                stops[i].record()
        barrier()
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, last)
    del last
    n_pairs = 1 if back_to_back else args.steps
    total_ms = max_over_ranks(sum(s.elapsed_time(e) for s, e in zip(starts[:n_pairs], stops[:n_pairs])))
    launches = pipe.launch_count() - launches0
    value = world * batch * nvox * passes * args.steps / (total_ms * 1e-3)

    # ---- one tensor at a time, stage profiler on: latency and the per-stage rooflines ----------------------
    p_steps = args.steps
    p_starts = [torch.cuda.Event(enable_timing=True) for _ in range(p_steps)]
    p_stops = [torch.cuda.Event(enable_timing=True) for _ in range(p_steps)]
    ctx.profile(True)
    ctx.stage_times(reset=True)
    ctx.stat("eig_flops", reset=True)
    barrier()
    for i in range(p_steps):
        flush_buf.fill_(i & 0xFF)
        p_starts[i].record()
        unit(vols[i % n_distinct])
        p_stops[i].record()
    barrier()
    single_ms = sum(s.elapsed_time(e) for s, e in zip(p_starts, p_stops)) / p_steps
    stages = ctx.stage_times(reset=True)
    eig_flops = ctx.stat("eig_flops", reset=True) / p_steps
    ctx.profile(False)

    # ---- end to end from pinned host buffers, same batch, same concurrency -----------------------------------
    h2d = batch * nvox * 4
    if workload == "cfg3":
        srcs = [pinned[i % n_distinct].numpy() for i in range(batch)]
        n_dst = min(batch, 2 * in_flight)
        dst_t = [torch.empty(shape, dtype=torch.float32).pin_memory() for _ in range(n_dst)]
        dsts = [dst_t[i % n_dst].numpy() for i in range(batch)]
        d2h = batch * nvox * 4
        entry = "VolumePipeline.roundtrip_host -> ndmps_roundtrip_host (C ABI, pinned host buffers)"

        def e2e_step(k=1):
            pipe.roundtrip_host(srcs * k, dsts * k, max_bond=chi)
    else:
        returns_rec = workload == "cfg5b"
        n_dst = min(batch, 2 * in_flight)
        dst_t = [torch.empty(shape, dtype=torch.float32).pin_memory() for _ in range(n_dst)] if returns_rec else []
        d2h = batch * nvox * 4 if returns_rec else batch * 8 * (2 if workload == "cfg1" else (3 * len(CHI_SWEEP) if workload == "cfg2" else 1))
        entry = "NDMPS.from_tensor(pinned host tensor -> device copy inside) + to_tensor + metrics; scalars" + (
            " and the reconstruction" if returns_rec else "") + " copied back"

        def one_host(j):
            v = pinned[j % n_distinct].cuda(non_blocking=True)
            rec_j, scal = unit(v)
            if returns_rec:
                dst_t[j % n_dst].copy_(rec_j, non_blocking=True)
            return scal

        def e2e_step(k=1):
            pipe.map(one_host, list(range(batch)) * k)
    for _ in range(3):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    if back_to_back:
        e2e_step(args.steps)                 # K steps = one queue of K x batch tensors: item i -> worker i mod in_flight
    else:
        for _ in range(args.steps):
            e2e_step()
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = world * batch * nvox * passes * args.steps / e2e_s
    e2e_err = None
    if workload == "cfg3":
        src, dst = srcs[0], dsts[0]
        e2e_err = float(np.linalg.norm(dst.astype(np.float64) - src) / np.linalg.norm(src.astype(np.float64)))
    pipe.close()

    # ---- N > 1 on the north-star volume: ONE volume column-sharded over the ranks (NCCL Gram allreduce) --------
    sharded = None
    if world > 1 and workload == "cfg3" and not args.no_sharded:
        sharded = sharded_volume_record(args, chi, torch, dist, ctx, flush_buf, world, rank, local)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- rooflines of the stages (algorithmic work / measured device time of the single-tensor pass) ---------
    peaks = load_peaks()
    fp64_tflops = measure_fp64_rate(torch)
    per_call = {k: (v[0] / p_steps, v[1] / p_steps) for k, v in stages.items()}
    work = work_for(workload, info, nvox)
    used_tc = bool(ctx.stat("tc_launches")) if _has_stat(ctx, "tc_launches") else False
    from imgcompressionmps import _ops as _ops_mod
    bit_permute = bool(_ops_mod.plan_for(tuple(WORKLOADS[workload]["shape"])).bit_info(False)["bits"])
    rooflines = build_rooflines(per_call, single_ms, work, nvox, peaks, fp64_tflops, eig_flops, used_tc, bit_permute)
    shares = {k: round(v[0] / single_ms, 4) for k, v in per_call.items() if v[1]}
    dominant = max(shares, key=shares.get) if shares else None
    roof = dict(rooflines.get(dominant) or {})
    roof.update({"peak_source": peaks["source"], "dominant_stage_by_time": dominant, "stage_share_of_tensor_time": shares,
                 "fp64_tflops_measured_in_run": fp64_tflops, "all": rooflines,
                 "note": "top level = the stage with the largest share of one tensor's time (single pass, stage profiler); "
                         "`all` has every stage"})
    hbm_floor_ms = (work["encode_bytes"] + work["decode_bytes"] + work["sweep_bytes"] + work["recon_bytes"] + work.get("metric_bytes", 0.0)) / (peaks["hbm_gbs"] * 1e6)
    result = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(workload, args, world),
        "run": {"tensors_per_step_per_gpu": batch, "tensors_in_flight_per_gpu": in_flight, "l2_flush_between_steps": not back_to_back,
                "steps_back_to_back": back_to_back,
                "l2_note": (f"the {n_distinct} distinct inputs of a step ({n_distinct * nvox * 4 / 1e6:.0f} MB) exceed the 126 MB L2 several times; "
                            "the K steps run back to back inside one event pair (value) / one host-clock bracket (e2e)") if back_to_back
                else "a 512 MB buffer is rewritten between steps, outside the per-step event pairs",
                "site_dims": info["site_dims"], "bond_dims": info["bond_dims"],
                "parallelism": f"{world} GPU(s) x {batch} independent tensors per step, {in_flight} in flight per GPU "
                               f"(host threads x CUDA streams), no data-path collective",
                "reconstruction_rel_error_vs_input": err,
                "scalars_of_first_tensor": {k: v for k, v in info.items() if k not in ("site_dims", "bond_dims")}},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1e3 * e2e_s / args.steps, "entry": entry, "reconstruction_rel_error_vs_input": e2e_err},
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
        "roofline": roof,
        "single": {"ms": single_ms, "value": nvox * passes / (single_ms * 1e-3), "unit": UNIT, "steps": p_steps,
                   "note": "one tensor at a time on one stream (latency); stage times and rooflines are from this pass",
                   "stage_ms": {k: round(v[0], 4) for k, v in per_call.items() if v[1]}},
        "speed_of_light": {"hbm_floor_ms_per_tensor": hbm_floor_ms, "hbm_floor_voxels_per_s": nvox * passes / (hbm_floor_ms * 1e-3),
                           "note": "SURVEY 8(d) algorithmic bytes / measured HBM peak"},
    }
    if sharded is not None:
        result["sharded"] = sharded
    if keep is not None:
        result["run"]["dump_outputs"] = {
            "dir": args.dump_outputs, "voxels_kept_per_tensor": int(keep.numel()),
            "note": "the last timed step also gathered the kept voxels of every reconstruction (one small kernel per tensor)"}
    if world == 1 and not args.no_cpu:
        rate, per, n_run = time_oracle(workload, chi, hosts[0], 1, 0.0)
        result["cpu_baseline"] = {
            "value": rate, "unit": UNIT, "cores": host_threads(), "kind": "port",
            "sample": f"one tensor of the workload ({'x'.join(map(str, shape))} float32, the same array the GPU arm's first slot holds), "
                      f"same unit of work on the oracle, numpy/LAPACK float64, one run ({per:.1f} s)"}
    print(json.dumps(result))
    if world > 1:
        dist.destroy_process_group()


def _has_stat(ctx, name):
    try:
        ctx.stat(name)
        return True
    except Exception:
        return False


def sharded_volume_record(args, chi, torch, dist, ctx, flush_buf, world, rank, local):
    """ONE 512^3 volume spread over the ranks (SURVEY section 8e row 2, BASELINE configs[2]): every rank holds the
    sub-lattice of the volume that forms a column block of the unfoldings, the sweep allreduces the bond-sized
    Gram matrix of every step over NCCL, the reconstruction stays sharded.  Strong scaling; returns the record
    rank 0 embeds in the JSON line (None elsewhere)."""
    from imgcompressionmps.distributed import ShardedNDMPS, shard_volume
    from imgcompressionmps.utils.core import get_factorlist

    shape = WORKLOADS["cfg3"]["shape"]
    nvox = int(np.prod(shape))
    factors, _ = get_factorlist(shape)
    host_local = np.ascontiguousarray(shard_volume(synthetic_volume(shape, 2027), factors, rank, world))   # cut at load time
    pinned = torch.from_numpy(host_local).pin_memory()
    out_pinned = torch.empty_like(pinned).pin_memory()
    vol = pinned.cuda()
    stats = {"calls": 0, "bytes": 0}

    def step(v):
        obj = ShardedNDMPS.from_local(v, shape, rank=rank, world=world, max_bond=chi)
        return obj, obj.to_local_tensor_device()

    for _ in range(3):
        obj, rec = step(vol)
    err2 = torch.stack([((rec - vol).double() ** 2).sum(), (vol.double() ** 2).sum()])
    if world > 1:
        dist.all_reduce(err2)
    err = float(torch.sqrt(err2[0] / err2[1]))
    steps = args.steps
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    launches0 = ctx.launch_count()
    if hasattr(ShardedNDMPS, "allreduce_stats"):
        ShardedNDMPS.allreduce_stats(reset=True)
    dist.barrier()
    torch.cuda.synchronize()
    for i in range(steps):
        flush_buf.fill_(i & 0xFF)
        starts[i].record()
        step(vol)
        stops[i].record()
    dist.barrier()
    torch.cuda.synchronize()
    if hasattr(ShardedNDMPS, "allreduce_stats"):
        stats = ShardedNDMPS.allreduce_stats(reset=True)
    t = torch.tensor([sum(s.elapsed_time(e) for s, e in zip(starts, stops))], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    launches = ctx.launch_count() - launches0
    t0 = time.perf_counter()
    for _ in range(steps):
        v = pinned.cuda(non_blocking=True)
        _, r = step(v)
        out_pinned.copy_(r, non_blocking=True)
        torch.cuda.synchronize()
    e2e = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    dist.all_reduce(e2e, op=dist.ReduceOp.MAX)
    if rank != 0:
        return None
    return {"what": f"ONE {'x'.join(map(str, shape))} volume column-sharded over {world} GPUs: local Gram + NCCL allreduce of the bond-sized "
                    "float64 Gram matrix per sweep step, replicated eigensolve, local projection, sharded reconstruction",
            "scaling": "strong", "n_gpus": world, "nccl_ranks": dist.get_world_size(), "steps": steps,
            "ms_per_volume": total_ms / steps, "value": nvox * steps / (total_ms * 1e-3), "unit": UNIT,
            "e2e_value": nvox * steps / float(e2e.item()), "e2e_ms_per_volume": 1e3 * float(e2e.item()) / steps,
            "bond_dims": obj.bond_sizes(), "reconstruction_rel_error_vs_input": err,
            "allreduce_calls_per_volume": stats.get("calls", 0) / steps if steps else 0,
            "allreduce_bytes_per_volume": stats.get("bytes", 0) / steps if steps else 0,
            "allreduce_ms_per_volume": stats.get("ms", 0.0) / steps if steps and stats.get("ms") is not None else None,
            "gpu_launches_per_volume_per_rank": launches / steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of every record; --impl reference stops sooner when --ref-budget runs out and "
                         "reports the steps it ran")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--chi", type=int, default=0, help="bond cap (0: the workload's own)")
    ap.add_argument("--in-flight", type=int, default=0, help="tensors processed concurrently per GPU (0: workload default)")
    ap.add_argument("--volumes", type=int, default=0, help="tensors per step per GPU (0: workload default)")
    ap.add_argument("--no-sharded", action="store_true", help="N > 1: skip the column-sharded single-volume record")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--per-step", action="store_true", help="one event pair and an L2 flush per step (drains the pipeline between steps)")
    ap.add_argument("--ref-budget", type=float, default=150.0, help="--impl reference: seconds of timed oracle work")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write what the last one computed (rank 0) as DIR/<name>.npy, at most 64 MB: "
                         "each tensor's reconstruction (a fixed seeded sample of its voxels when the step's are too many) "
                         "and the unit's scalars and bond dimensions")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload == "cfg5"):
        ap.error("--dump-outputs needs --impl ours and a timed workload (not cfg5)")
    if args.workload == "cfg5":
        if int(os.environ.get("RANK", "0")) == 0:
            degenerate_report(args)
        return
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
