#!/usr/bin/env python
"""Maximum-intensity projections from the cores against the reconstruction followed by torch.amax, on the device.

Workloads:
  config 3 - one 512^3 float32 phantom (bench.synthetic_volume) at chi = 64, mode Std:
    project_device(a) for a = 0, 1, 2 (baseline to_tensor_device().amax(a)) and a 40-slice thick-slab MIP,
    project_device(0, index=(slice(z, z + 40),)) (baseline to_tensor_region_device(slab).amax(0));
  config 5-B - one (1920, 1080, 64) float32 DCT video chunk (bench.synthetic_video) at chi = 64:
    the max over frames (the last axis) and along axis 0.
Calls are warmed up, then timed with CUDA events around `--reps` calls (median and min reported), with the peak torch
allocation of one more call.  The projections run in a thread of their own, so the library workspace high-water mark
recorded after each of them belongs to the projection path alone.  The card's name and power limit are recorded beside
the numbers.

    python tools/project_probe.py --out project_probe.json
"""
import argparse
import json
import sys
import threading
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
for p in (str(ROOT), str(ROOT / "img-compression-mps_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
from bench import synthetic_video, synthetic_volume     # noqa: E402
from imgcompressionmps.core.ndmps import NDMPS          # noqa: E402
from probe_timing import card, timed                    # noqa: E402


def probe(obj, cases, reps, warmup):
    """cases: (name, axis, index).  Projections in a fresh thread (own context and arena), baselines here."""
    from imgcompressionmps import _native
    rows, outs, err = [], {}, []

    def project_side():
        try:
            for name, axis, index in cases:
                out, rec = timed(lambda: obj.project_device(axis, "max", index), reps, warmup)
                torch.cuda.synchronize()
                rec.update(name=name, axis=axis, out_shape=list(out.shape), path="project_device",
                           workspace_high_water_MB=_native.context().stat("workspace_bytes") / 2 ** 20)
                outs[name] = out
                rows.append(rec)
                print(json.dumps(rec), flush=True)
        except Exception as exc:                        # surfaced below
            err.append(exc)

    t = threading.Thread(target=project_side)
    t.start()
    t.join()
    if err:
        raise err[0]
    for name, axis, index in cases:
        def baseline():
            rec = obj.to_tensor_device() if index is None else obj.to_tensor_region_device(index)
            return rec.amax(dim=axis)

        ref, rec = timed(baseline, reps, warmup)
        rec.update(name=name, axis=axis, path="to_tensor_device() + amax" if index is None
                   else "to_tensor_region_device(slab) + amax")
        got = outs[name]
        rec["project_max_abs_diff"] = float((got.double() - ref.double()).abs().max())
        rec["project_max_abs_diff_rel_to_max"] = rec["project_max_abs_diff"] / float(ref.double().abs().max())
        rec["project_matches_baseline"] = rec["project_max_abs_diff_rel_to_max"] <= 1e-5
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
    assert torch.cuda.is_available(), "project_probe measures on the GPU; there is no CPU path"
    torch.cuda.set_device(0)
    report = {"card": card(), "timing": "CUDA events around each call, after warm-up; median of --reps calls"}

    n = args.n
    vol = torch.from_numpy(synthetic_volume((n, n, n), 2027)).cuda()
    obj = NDMPS.from_tensor(vol, max_bond=64)
    del vol
    z = n // 2 - 20
    cases = [(f"MIP axis {a}", a, None) for a in range(3)] + [(f"40-slice slab MIP, slices {z}..{z + 39}", 0,
                                                                (slice(z, z + 40),))]
    report["config3"] = {"shape": [n] * 3, "chi": 64, "bonds": obj.bond_sizes(),
                         "rows": probe(obj, cases, args.reps, args.warmup)}
    del obj
    torch.cuda.empty_cache()

    if args.video:
        shape = tuple(int(v) for v in args.video.split(","))
        vid = torch.from_numpy(synthetic_video(shape, 4000)).cuda()
        obj = NDMPS.from_tensor(vid, mode="DCT", max_bond=64)
        del vid
        cases = [("max over frames (axis 2)", 2, None), ("max along axis 0", 0, None)]
        report["config5b"] = {"shape": list(shape), "chi": 64, "mode": "DCT", "bonds": obj.bond_sizes(),
                              "rows": probe(obj, cases, args.reps, args.warmup)}
    report["all_match"] = all(r["project_matches_baseline"] for cfg in ("config3", "config5b") if cfg in report
                              for r in report[cfg]["rows"] if "project_matches_baseline" in r)
    text = json.dumps(report, indent=1)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
