#!/usr/bin/env python
"""Block-mean (coarse) decode against the full reconstruction followed by a block mean, on the device.

Workloads:
  config 3 - one 512^3 float32 phantom (bench.synthetic_volume) at chi = 64, mode Std:
    to_tensor_coarse_device(k) for k = 1, 2, 3 (256^3, 128^3, 64^3) and one slice of the k = 2 result;
  config 5-B - one (1920, 1080, 64) float32 DCT video chunk (bench.synthetic_video) at chi = 64:
    levels (1, 1, 0), (2, 2, 0) and (1, 1, 1).
Each case is timed beside its baseline, to_tensor_device() followed by a torch block mean, and its output is compared
with that baseline.  Calls are warmed up, then timed with CUDA events around `--reps` calls (median and min
reported), with the peak torch allocation of one more call.  The coarse calls run in a thread of their own, so the
library workspace high-water mark recorded after each of them belongs to the coarse path alone.  The card's name and
power limit are recorded beside the numbers.

    python tools/coarse_probe.py --out coarse_probe.json
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


def block_mean(x, block):
    split = []
    for s, b in zip(x.shape, block):
        split += [s // b, b]
    return x.view(split).mean(dim=tuple(range(1, 2 * x.dim(), 2)))


def probe(obj, cases, reps, warmup):
    """cases: (name, levels, index).  Coarse calls in a fresh thread (own context and arena), baselines here."""
    from imgcompressionmps import _native
    rows, outs, err = [], {}, []

    def coarse_side():
        try:
            for name, levels, index in cases:
                out, rec = timed(lambda: obj.to_tensor_coarse_device(levels, index), reps, warmup)
                torch.cuda.synchronize()
                rec.update(name=name, levels=levels, coarse_shape=list(obj.coarse_shape(levels)), path="coarse",
                           workspace_high_water_MB=_native.context().stat("workspace_bytes") / 2 ** 20)
                outs[name] = out
                rows.append(rec)
                print(json.dumps(rec), flush=True)
        except Exception as exc:                        # surfaced below
            err.append(exc)

    t = threading.Thread(target=coarse_side)
    t.start()
    t.join()
    if err:
        raise err[0]
    for name, levels, index in cases:
        block = tuple(s // c for s, c in zip(obj.shape, obj.coarse_shape(levels)))

        def baseline():
            m = block_mean(obj.to_tensor_device(), block)
            return m if index is None else m[index]

        ref, rec = timed(baseline, reps, warmup)
        rec.update(name=name, levels=levels, path="to_tensor_device() + block mean")
        got = outs[name]
        rec["coarse_max_abs_err_rel_to_max"] = float((got.double() - ref.double()).abs().max() / ref.double().abs().max())
        rec["coarse_matches_baseline"] = rec["coarse_max_abs_err_rel_to_max"] <= 1e-5
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
    assert torch.cuda.is_available(), "coarse_probe measures on the GPU; there is no CPU path"
    torch.cuda.set_device(0)
    report = {"card": card(), "timing": "CUDA events around each call, after warm-up; median of --reps calls"}

    n = args.n
    vol = torch.from_numpy(synthetic_volume((n, n, n), 2027)).cuda()
    obj = NDMPS.from_tensor(vol, max_bond=64)
    del vol
    z = obj.coarse_shape(2)[0] // 2
    cases = [("levels 1", 1, None), ("levels 2", 2, None), ("levels 3", 3, None), ("levels 2, slice (z,)", 2, (z,))]
    report["config3"] = {"shape": [n] * 3, "chi": 64, "bonds": obj.bond_sizes(),
                         "rows": probe(obj, cases, args.reps, args.warmup)}
    del obj
    torch.cuda.empty_cache()

    if args.video:
        shape = tuple(int(v) for v in args.video.split(","))
        vid = torch.from_numpy(synthetic_video(shape, 4000)).cuda()
        obj = NDMPS.from_tensor(vid, mode="DCT", max_bond=64)
        del vid
        cases = [(f"levels {k}", k, None) for k in ((1, 1, 0), (2, 2, 0), (1, 1, 1))]
        report["config5b"] = {"shape": list(shape), "chi": 64, "mode": "DCT", "bonds": obj.bond_sizes(),
                              "rows": probe(obj, cases, args.reps, args.warmup)}
    report["all_match"] = all(r["coarse_matches_baseline"] for cfg in ("config3", "config5b") if cfg in report
                              for r in report[cfg]["rows"] if "coarse_matches_baseline" in r)
    text = json.dumps(report, indent=1)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
