#!/usr/bin/env python
"""Interpolated sampling from the cores against the full reconstruction followed by torch's grid_sample, on the device.

Workloads (float32, mode Std, chi = 64):
  plane    - one 512^3 phantom (config 3, bench.synthetic_volume): a 512 x 512 oblique plane through the centre,
             spanned by u = (1, 1, 0)/sqrt(2) and v = (1, -1, 1)/sqrt(3) at one voxel per sample (corners clamp);
             sample_grid_device, and sample() with the same coordinates as a float64 device array;
  resample - one 256^3 phantom resampled to 200^3 with the corners kept: sample_grid_device.
The baseline is to_tensor_device() followed by torch.nn.functional.grid_sample(mode="bilinear", align_corners=True,
padding_mode="border") on a normalised grid built before the timed window (so the baseline is not charged for it).
Calls are warmed up, then timed with CUDA events around `--reps` calls (median and min reported), with the peak torch
allocation of one more call.  The sampling calls run in a thread of their own, so the library workspace high-water
mark recorded after them belongs to the sampling path alone.  Outputs are compared with the baseline's.  The card's
name and power limit are recorded beside the numbers.

    python tools/sample_probe.py --out-dir probe_out
"""
import argparse
import json
import sys
import threading
from pathlib import Path

import numpy as np
import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parents[1]
for p in (str(ROOT), str(ROOT / "img-compression-mps_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
from bench import synthetic_volume                      # noqa: E402
from imgcompressionmps.core.ndmps import NDMPS          # noqa: E402
from probe_timing import card, timed                    # noqa: E402


def normalised_grid(origin, steps, out_shape, shape):
    """grid_sample's grid (1, *out_shape, 3) for the coordinates origin + sum_j i_j steps[j] of a (D, H, W) volume:
    the last dimension is (w, h, d), each mapped to [-1, 1] with the corners aligned."""
    idx = torch.stack(torch.meshgrid(*[torch.arange(n, dtype=torch.float64, device="cuda") for n in out_shape],
                                     indexing="ij"), dim=-1)
    c = torch.as_tensor(origin, device="cuda") + idx @ torch.as_tensor(np.asarray(steps), device="cuda")
    ext = torch.tensor(shape, dtype=torch.float64, device="cuda")
    g = (2.0 * c / (ext - 1) - 1.0).flip(-1)
    return g.to(torch.float32).reshape(1, *([1] * (3 - len(out_shape))), *out_shape, 3), c.reshape(-1, 3).contiguous()


def probe(obj, cases, reps, warmup):
    """cases: (name, origin, steps, out_shape).  Sampling calls in a fresh thread (own context and arena), then the
    baselines here."""
    from imgcompressionmps import _native
    rows, outs, err = [], {}, []
    grids = {name: normalised_grid(o, s, m, obj.shape) for name, o, s, m in cases}

    def sample_side():
        try:
            for name, origin, steps, out_shape in cases:
                out, rec = timed(lambda: obj.sample_grid_device(origin, steps, out_shape), reps, warmup)
                rec.update(name=name, path="sample_grid_device", out_shape=list(out_shape),
                           workspace_high_water_MB=_native.context().stat("workspace_bytes") / 2 ** 20)
                outs[name] = out
                rows.append(rec)
                print(json.dumps(rec), flush=True)
                coords = grids[name][1]
                pts, rec = timed(lambda: obj.sample(coords), reps, warmup)
                rec.update(name=name, path="sample(float64 device coordinates)", out_shape=list(out_shape),
                           coords_MB=coords.numel() * 8 / 2 ** 20,
                           max_abs_diff_to_grid=float((pts.view(out.shape).double() - out.double()).abs().max()))
                rows.append(rec)
                print(json.dumps(rec), flush=True)
        except Exception as exc:                        # surfaced below
            err.append(exc)

    t = threading.Thread(target=sample_side)
    t.start()
    t.join()
    if err:
        raise err[0]
    for name, origin, steps, out_shape in cases:
        grid = grids[name][0]

        def baseline():
            rec = obj.to_tensor_device()
            return F.grid_sample(rec[None, None], grid, mode="bilinear", padding_mode="border", align_corners=True)

        ref, rec = timed(baseline, reps, warmup)
        rec.update(name=name, path="to_tensor_device() + grid_sample", out_shape=list(out_shape),
                   grid_MB=grid.numel() * 4 / 2 ** 20)
        got = outs[name].reshape(-1).double()
        ref = ref.reshape(-1).double()
        rec["sample_max_abs_err_rel_to_max"] = float((got - ref).abs().max() / ref.abs().max())
        rows.append(rec)
        print(json.dumps(rec), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--n", type=int, default=512, help="edge of the config-3 cube of the plane workload")
    ap.add_argument("--resample", default="256,200", help="edge of the resampled cube and of its output")
    ap.add_argument("--out-dir", required=True, help="directory the JSON report is written to")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "sample_probe measures on the GPU; there is no CPU path"
    torch.cuda.set_device(0)
    report = {"card": card(), "timing": "CUDA events around each call, after warm-up; median of --reps calls"}

    n = args.n
    vol = torch.from_numpy(synthetic_volume((n, n, n), 2027)).cuda()
    obj = NDMPS.from_tensor(vol, max_bond=64)
    del vol
    u = np.array([1.0, 1.0, 0.0]) / np.sqrt(2.0)
    v = np.array([1.0, -1.0, 1.0]) / np.sqrt(3.0)
    half = (n - 1) / 2.0
    plane = ("oblique plane", np.full(3, half) - half * (u + v), np.stack([u, v]), (n, n))
    report["plane"] = {"shape": [n] * 3, "chi": 64, "bonds": obj.bond_sizes(),
                       "multiply_adds_per_sample": 8 * max(obj.bond_sizes()),
                       "rows": probe(obj, [plane], args.reps, args.warmup)}
    del obj
    torch.cuda.empty_cache()

    m, k = (int(x) for x in args.resample.split(","))
    vol = torch.from_numpy(synthetic_volume((m, m, m), 2028)).cuda()
    obj = NDMPS.from_tensor(vol, max_bond=64)
    del vol
    resample = ("resample", np.zeros(3), np.eye(3) * (m - 1) / (k - 1), (k, k, k))
    report["resample"] = {"shape": [m] * 3, "out_shape": [k] * 3, "chi": 64, "bonds": obj.bond_sizes(),
                          "rows": probe(obj, [resample], args.reps, args.warmup)}
    text = json.dumps(report, indent=1)
    out = Path(args.out_dir)
    out.mkdir(parents=True, exist_ok=True)
    (out / "sample_probe.json").write_text(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
