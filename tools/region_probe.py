#!/usr/bin/env python
"""Box decode and point evaluation against the full reconstruction, on the device.

Workloads:
  config 3 - one 512^3 float32 phantom (bench.synthetic_volume) at chi = 64, mode Std:
    to_tensor_device(), to_tensor()[z], one slice on each axis, an aligned 128^3 box, an unaligned 100^3 box,
    values_at with 10^4 and 10^6 random points (CUDA coordinates);
  config 5-B - one (1920, 1080, 64) float32 DCT video chunk (bench.synthetic_video) at chi = 64:
    to_tensor_device(), one frame (last axis an int: decoded over all 64 frames, then inverse DCT, then cropped),
    a 256 x 256 spatial crop (all 64 frames), values_at with 10^4 and 10^6 random points (CUDA coordinates; each
    point sums the 64 coefficients of its line).
Each call is warmed up, then timed with CUDA events around `--reps` calls (median and min reported), and its output
is compared with the same part of the full reconstruction.  Peak torch allocation per call and the library's
workspace high-water mark are recorded beside the times, with the card's name and power limit.

    python tools/region_probe.py --out region_probe.json
"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
for p in (str(ROOT), str(ROOT / "img-compression-mps_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
from bench import synthetic_video, synthetic_volume     # noqa: E402
from imgcompressionmps.core.ndmps import NDMPS          # noqa: E402
from probe_timing import card, timed                    # noqa: E402


def rel_err(got, want):
    got = got if isinstance(got, torch.Tensor) else torch.as_tensor(got)
    got = got.to(want.device, torch.float64)
    return float((got - want.double()).abs().max() / want.double().abs().max())


def random_points(shape, seed):
    """10^4 and 10^6 seeded random points of a volume of ``shape``, as CUDA int64 (K, ndim) tensors."""
    rng = np.random.default_rng(seed)
    return {k: torch.as_tensor(np.stack([rng.integers(0, n, size=k) for n in shape], axis=1), device="cuda")
            for k in (10 ** 4, 10 ** 6)}


def probe(obj, full, items, reps, warmup):
    rows = []
    for name, fn, ref in items:
        out, rec = timed(fn, reps, warmup)
        rec["name"] = name
        if ref is not None:
            rec["max_abs_err_rel_to_max"] = rel_err(out, ref())
        rows.append(rec)
        print(json.dumps(rec), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--n", type=int, default=512, help="edge of the config-3 cube")
    ap.add_argument("--video", default="1920,1080,64", help="shape of the config 5-B chunk ('' skips it)")
    ap.add_argument("--out", default=None, help="write the JSON report here")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "region_probe measures on the GPU; there is no CPU path"
    torch.cuda.set_device(0)
    from imgcompressionmps import _native
    report = {"card": card(), "timing": "CUDA events around each call, after warm-up; median of --reps calls"}

    n = args.n
    vol = torch.from_numpy(synthetic_volume((n, n, n), 2027)).cuda()
    obj = NDMPS.from_tensor(vol, max_bond=64)
    del vol
    full = obj.to_tensor_device()
    z, c = n // 2, n // 4
    pts = random_points((n, n, n), 5)
    items = [
        ("to_tensor_device()", obj.to_tensor_device, None),
        ("to_tensor()[z]", lambda: obj.to_tensor()[z], lambda: full[z]),
        ("region (z,) axis 0 slice", lambda: obj.to_tensor_region_device((z,)), lambda: full[z]),
        ("region (:, z) axis 1 slice", lambda: obj.to_tensor_region_device((slice(None), z)), lambda: full[:, z]),
        ("region (..., z) axis 2 slice", lambda: obj.to_tensor_region_device((Ellipsis, z)), lambda: full[..., z]),
        ("region 128^3 aligned", lambda: obj.to_tensor_region_device((slice(c, c + 128),) * 3),
         lambda: full[c:c + 128, c:c + 128, c:c + 128]),
        ("region 100^3 unaligned", lambda: obj.to_tensor_region_device((slice(c + 37, c + 137),) * 3),
         lambda: full[c + 37:c + 137, c + 37:c + 137, c + 37:c + 137]),
    ] + [(f"values_at {k} points", lambda k=k: obj.values_at(pts[k]), lambda k=k: full[tuple(pts[k].T)]) for k in pts]
    report["config3"] = {"shape": [n] * 3, "chi": 64, "bonds": obj.bond_sizes(),
                         "rows": probe(obj, full, items, args.reps, args.warmup)}
    del obj, full
    torch.cuda.empty_cache()

    if args.video:
        shape = tuple(int(v) for v in args.video.split(","))
        vid = torch.from_numpy(synthetic_video(shape, 4000)).cuda()
        obj = NDMPS.from_tensor(vid, mode="DCT", max_bond=64)
        del vid
        full = obj.to_tensor_device()
        f = shape[2] // 3
        x0, y0 = shape[0] // 2 - 128, shape[1] // 2 - 128
        pts = random_points(shape, 6)
        items = [
            ("to_tensor_device()", obj.to_tensor_device, None),
            ("region (..., f) one frame", lambda: obj.to_tensor_region_device((Ellipsis, f)), lambda: full[..., f]),
            ("region 256x256 crop, all frames", lambda: obj.to_tensor_region_device((slice(x0, x0 + 256), slice(y0, y0 + 256))),
             lambda: full[x0:x0 + 256, y0:y0 + 256]),
        ] + [(f"values_at {k} points", lambda k=k: obj.values_at(pts[k]), lambda k=k: full[tuple(pts[k].T)]) for k in pts]
        report["config5b"] = {"shape": list(shape), "chi": 64, "mode": "DCT", "bonds": obj.bond_sizes(),
                              "rows": probe(obj, full, items, args.reps, args.warmup)}
    report["workspace_high_water_MB"] = _native.context().stat("workspace_bytes") / 2 ** 20
    text = json.dumps(report, indent=1)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
