"""The JSON line of bench.py's reference arm (the CPU leg runs anywhere) carries the keys the driver reads."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]


def test_reference_arm_line():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "cfg1", "--steps", "2",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["value"] > 0 and d["unit"] == "voxels/s"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]
    # both arms print the SAME config object: it is a function of the command line only
    sys.path.insert(0, str(ROOT))
    import argparse

    import bench
    args = argparse.Namespace(chi=0)
    assert d["config"] == bench.workload_config("cfg1", args, 1)
    assert bench.workload_config("cfg3", args, 1)["shape"] == [512, 512, 512]


def test_default_workload_is_the_north_star_volume_and_cfg5_is_reported_degenerate():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "cfg5"], capture_output=True, text=True, timeout=300,
                         cwd=str(ROOT))
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][0])
    assert d["degenerate"]["levels"] == 1 and d["degenerate"]["site_dims"] == [1920 * 1080 * 3 * 512] and d["degenerate"]["bonds"] == []
    sys.path.insert(0, str(ROOT))
    import bench
    src = (ROOT / "bench.py").read_text()
    assert 'ap.add_argument("--workload", default="cfg3"' in src
    assert bench.WORKLOADS["cfg3"]["shape"] == (512, 512, 512) and bench.WORKLOADS["cfg3"]["chi"] == 64


def test_algorithmic_work_matches_survey_table():
    """SURVEY section 8(d): 256^3 at chi = 64 -> 70.9 bytes/voxel and 1895 flop/voxel for encode + sweep + reconstruct + decode."""
    sys.path.insert(0, str(ROOT))
    import bench
    dims, ranks = [8] * 8, [8, 64, 64, 64, 64, 64, 8]
    w = bench.algorithmic_work(dims, ranks)
    n = 8 ** 8
    bytes_per_voxel = (w["encode_bytes"] + w["decode_bytes"] + w["sweep_bytes"] + w["recon_bytes"]) / n
    flops_per_voxel = (w["gram_flops"] + w["project_flops"] + w["recon_flops"]) / n
    assert abs(bytes_per_voxel - 70.9) < 0.2
    assert abs(flops_per_voxel - 1895) < 5
    assert w["gram_flops_issued"] < w["gram_flops_executed"]


def test_roofline_entries_follow_the_contract():
    """Every stage entry: ``bound`` from the contract's enum, ``frac`` = achieved / peak, ``traffic`` read from an ncu CSV
    committed under profiles/ (the row of the kernel that really runs the stage), algorithmic figures beside it."""
    import bench
    info = {"site_dims": [8] * 9, "bond_dims": [8, 37, 64, 64, 64, 64, 64, 8]}
    nvox = 512 ** 3
    work = bench.work_for("cfg3", info, nvox)
    per_call = {"permute": (0.36, 2), "gram": (1.0, 6), "eig": (8.2, 8), "project": (0.32, 4), "contract": (0.23, 1)}
    peaks = {"hbm_gbs": 6559.4, "bf16_tflops": 1648.0}
    roof = bench.build_rooflines(per_call, 11.2, work, nvox, peaks, 35.3, 1.1e9, True, True)
    assert set(roof) == set(per_call)
    for stage, e in roof.items():
        assert e["bound"] in ("hbm", "tensor"), stage
        assert e["frac"] == pytest.approx(e["achieved"] / e["peak"])
        assert e["traffic"] and e["traffic_source"].startswith("profiles/r0"), stage
        assert e["share_of_tensor_time"] == pytest.approx(per_call[stage][0] / 11.2)
    # the permutation of a power-of-two volume is the register kernel: 2 x 8 B/voxel in 0.36 ms against the measured copy peak
    assert "permute_bits_kernel" in roof["permute"]["kernel"] and roof["permute"]["traffic_source"].endswith("r02b_kernels_raw.csv")
    assert roof["permute"]["algorithmic_bytes_per_tensor"] == 16 * nvox and roof["permute"]["frac"] == pytest.approx(0.909, abs=2e-3)
    # ncu's DRAM traffic of ONE launch (encode or decode: 8 B/voxel) = the algorithmic bytes of that launch
    assert roof["permute"]["calls_per_tensor"] == 2 and roof["permute"]["traffic"] == pytest.approx(8 * nvox, rel=0.06)
    assert "proj_i8_kernel" in roof["project"]["kernel"] and roof["project"]["traffic"] > 6e8
    assert "latency-bound" in roof["eig"]["bound_note"]
    tiles = bench.build_rooflines(per_call, 11.2, work, nvox, peaks, 35.3, 1.1e9, True, False)
    assert "permute_tiled_kernel" in tiles["permute"]["kernel"]


def test_dump_outputs_layout_and_size_limit(tmp_path):
    """--dump-outputs: the kept voxels are fixed by a seed, every workload's default step fits in 64 MB, and each
    output of the unit becomes one float32 / float64 .npy with the step's tensors along axis 0."""
    import numpy as np
    import torch

    import bench
    for key, wl in bench.WORKLOADS.items():
        pos = bench.dump_positions(int(np.prod(wl["shape"])), wl["batch"])
        assert 8 * wl["batch"] * pos.size <= bench.DUMP_LIMIT, key
        assert np.all(np.diff(pos) > 0) and np.array_equal(pos, bench.dump_positions(int(np.prod(wl["shape"])), wl["batch"]))
    assert np.array_equal(bench.dump_positions(1000, 4), np.arange(1000))
    rec = torch.arange(12, dtype=torch.float32)
    bench.write_outputs(tmp_path / "plain", [(rec + i, {"bond_dims": [8, 64, 8], "site_dims": [8, 8, 8, 8]}) for i in range(3)])
    got = {p.stem: np.load(p) for p in (tmp_path / "plain").iterdir() if p.suffix == ".npy"}
    assert sorted(p.name for p in (tmp_path / "plain").iterdir()) == ["bond_dims.npy", "reconstruction.npy", "site_dims.npy"]
    assert got["reconstruction"].dtype == np.float32 and got["reconstruction"].shape == (3, 12) and got["reconstruction"][2, 0] == 2
    assert got["bond_dims"].dtype == np.float64 and got["bond_dims"].tolist() == [[8, 64, 8]] * 3
    sweep = {"site_dims": [8] * 8, "bond_dims": {128: [8, 64], 8: [8, 8]}, "fidelity": {128: 1.0, 8: 0.9}, "psnr": {128: 50.0, 8: 30.0}}
    bench.write_outputs(tmp_path / "sweep", [(None, sweep)] * 2)
    assert sorted(p.name for p in (tmp_path / "sweep").iterdir()) == [
        "bond_dims_chi128.npy", "bond_dims_chi8.npy", "fidelity_chi128.npy", "fidelity_chi8.npy", "psnr_chi128.npy", "psnr_chi8.npy",
        "site_dims.npy"]
    with pytest.raises(SystemExit):
        bench.write_outputs(tmp_path / "big", [(torch.zeros(bench.DUMP_LIMIT // 4 + 1), {})])


@pytest.mark.gpu
def test_dump_outputs_hold_what_the_timed_path_computed(tmp_path):
    """bench.py --dump-outputs on the default workload: the kept voxels of the last timed step are those of the same
    volume reconstructed on its own, and the bond dimensions are the step's."""
    import numpy as np
    import torch

    import bench
    from imgcompressionmps.core.ndmps import NDMPS
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--volumes", "1", "--in-flight", "1", "--steps", "2", "--warmup", "1",
                          "--no-cpu", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=str(ROOT))
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][0])
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= bench.DUMP_LIMIT + 4096
    rec, bonds = np.load(tmp_path / "reconstruction.npy"), np.load(tmp_path / "bond_dims.npy")
    pos = bench.dump_positions(512 ** 3, 1)
    assert rec.shape == (1, pos.size) and rec.dtype == np.float32
    assert line["run"]["dump_outputs"]["voxels_kept_per_tensor"] == pos.size
    assert bonds.tolist() == [line["run"]["bond_dims"]]
    x = torch.from_numpy(bench.make_input("cfg3", 0, 0)).cuda()
    obj = NDMPS.from_tensor(x, max_bond=64)
    want = obj.to_tensor_device().reshape(-1)[torch.from_numpy(pos).cuda()].cpu().numpy()
    assert bonds.tolist() == [obj.bond_sizes()]
    assert np.linalg.norm(rec[0] - want) <= 1e-5 * np.linalg.norm(want)
