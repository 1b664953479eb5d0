"""The host-side orchestration of ``evaluation.benchmark``, checked the way the original project's own
``tests/evaluation/test_benchmark.py`` checks its module (SURVEY section 4, the row of that file): an
autouse fixture replaces ``NDMPS`` with a stand-in class, the three metric functions with constants and ``nib.load``
with a fake, all through the module's globals, so no GPU is needed.  What is pinned: one value per tensor from
``benchmark_metric`` for every metric name, the result layout of ``run_benchmark`` (``[tensor][level]``,
``bond_dims`` as ``[level][tensor]``), cumulative in-place compression, the JSON path handling and the result keys
of ``run_full_benchmark``, and the error types of every entry point."""
import json
from pathlib import Path

import numpy as np
import pytest

import imgcompressionmps.evaluation.benchmark as B

SSIM, PSNR, FIDELITY = 0.875, 31.5, 0.9375
METRICS = ["ssim", "compression_ratio", "bond_dims", "psnr", "fidelity", "storage", "gzip_bytes", "gzip_ratio", "shape"]


class _FakeNDMPS:
    """The methods the benchmark module calls, with values that tell the calls apart."""
    created = []

    def __init__(self, data, norm, mode, extras):
        self.data, self.norm, self.mode, self.extras, self.cuts = np.asarray(data), norm, mode, extras, []

    @classmethod
    def from_tensor(cls, data, norm=False, mode="DCT", **extras):
        obj = cls(data, norm, mode, extras)
        cls.created.append(obj)
        return obj

    def to_tensor(self):
        return self.data

    def compress(self, cutoff):
        self.cuts.append(cutoff)

    def compression_ratio(self):
        return 1.0 / (1 + len(self.cuts))

    def bond_sizes(self):
        return [2, 4 - len(self.cuts)]

    def get_storage_space(self, dtype):
        return 100.0 * np.dtype(dtype).itemsize

    def get_bytesize_on_disk(self, dtype=np.uint16):
        return 40 * np.dtype(dtype).itemsize

    def compression_ratio_on_disk(self, dtype=np.uint16, replace=False):
        assert replace is True
        return 0.5 / (1 + len(self.cuts))


class _FakeImage:
    def __init__(self, path):
        self.path = path
        self.header = self

    def get_fdata(self):
        return np.full((4, 6, 8), 2.0)

    def get_data_dtype(self):
        return np.dtype(np.int16)


class _FakeNib:
    loaded = []

    @classmethod
    def load(cls, path):
        cls.loaded.append(path)
        return _FakeImage(path)


@pytest.fixture(autouse=True)
def stand_ins(monkeypatch):
    _FakeNDMPS.created, _FakeNib.loaded = [], []
    monkeypatch.setattr(B, "NDMPS", _FakeNDMPS)
    monkeypatch.setattr(B, "nib", _FakeNib)
    monkeypatch.setattr(B, "compute_ssim_by_dim", lambda a, b: SSIM)
    monkeypatch.setattr(B, "compute_psnr", lambda a, b: PSNR)
    monkeypatch.setattr(B, "compute_overlap", lambda a, b: FIDELITY)


def _tensors(n=3):
    return [np.arange(24, dtype=np.float64).reshape(2, 3, 4) + i for i in range(n)]


def _mps(n=3):
    return [_FakeNDMPS.from_tensor(t) for t in _tensors(n)]


# ---- conv_to_mps / conv_to_tensors / compress_list --------------------------------------------------------------
def test_conv_to_mps_builds_one_object_per_tensor_with_norm_false(capsys):
    out = B.conv_to_mps(_tensors(), mode="Std")
    assert len(out) == 3 and all(isinstance(m, _FakeNDMPS) for m in out)
    assert all(m.norm is False and m.mode == "Std" and m.extras == {} for m in out)
    assert "Converting file 3/3" in capsys.readouterr().out


def test_conv_to_mps_default_mode_is_dct():
    assert B.conv_to_mps(_tensors(1))[0].mode == "DCT"


def test_conv_to_mps_empty_list():
    assert B.conv_to_mps([]) == []


def test_conv_to_tensors_returns_every_reconstruction(capsys):
    mps = _mps()
    out = B.conv_to_tensors(mps)
    assert all(np.array_equal(o, t) for o, t in zip(out, _tensors()))
    assert "Converting file 3/3" in capsys.readouterr().out


def test_conv_to_tensors_empty_list():
    assert B.conv_to_tensors([]) == []


def test_compress_list_compresses_every_item_in_place():
    mps = _mps()
    assert B.compress_list(mps, 0.25) is None
    assert [m.cuts for m in mps] == [[0.25]] * 3


def test_compress_list_rejects_none():
    with pytest.raises(ValueError):
        B.compress_list(_mps(), None)


# ---- benchmark_metric ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", METRICS)
def test_benchmark_metric_one_value_per_tensor(metric):
    mps, tensors = _mps(), _tensors()
    refs = {"ssim": tensors, "psnr": tensors, "shape": tensors, "fidelity": _mps()}.get(metric)
    got = B.benchmark_metric(mps, refs, metric=metric)
    want = {"ssim": SSIM, "psnr": PSNR, "fidelity": FIDELITY, "compression_ratio": 1.0, "bond_dims": [2, 4],
            "storage": 200.0, "gzip_bytes": 80, "gzip_ratio": 0.5, "shape": (2, 3, 4)}[metric]
    assert got == [want] * 3


def test_benchmark_metric_storage_follows_dtype():
    assert B.benchmark_metric(_mps(1), metric="storage", dtype=np.uint8) == [100.0]


def test_benchmark_metric_default_is_compression_ratio():
    assert B.benchmark_metric(_mps(2)) == [1.0, 1.0]


def test_benchmark_metric_rejects_unknown_names():
    with pytest.raises(ValueError):
        B.benchmark_metric(_mps(), metric="entropy")


def test_benchmark_metric_length_mismatch():
    with pytest.raises(IndexError):
        B.benchmark_metric(_mps(3), _tensors(2), metric="ssim")


def test_benchmark_metric_empty_list():
    assert B.benchmark_metric([], metric="ssim") == []


# ---- run_benchmark ---------------------------------------------------------------------------------------------
def test_run_benchmark_result_shapes_and_keys():
    res = B.run_benchmark(_mps(3), _tensors(3), [0.1, 0.2])
    assert set(res) == {"ssim", "compression_ratio", "bond_dims", "psnr", "fidelity", "storage", "gzip_bytes", "gzip_ratio"}
    for name in ("ssim", "compression_ratio", "psnr", "fidelity", "storage", "gzip_bytes", "gzip_ratio"):
        assert np.asarray(res[name]).shape == (3, 3), name


def test_run_benchmark_values_per_level():
    res = B.run_benchmark(_mps(2), _tensors(2), [0.1, 0.2])
    assert np.allclose(res["compression_ratio"], [[1.0, 0.5, 1 / 3]] * 2)
    assert np.allclose(res["gzip_ratio"], [[0.5, 0.25, 0.5 / 3]] * 2)
    assert np.allclose(res["ssim"], SSIM) and np.allclose(res["psnr"], PSNR) and np.allclose(res["fidelity"], FIDELITY)


def test_run_benchmark_bond_dims_are_level_major():
    res = B.run_benchmark(_mps(2), _tensors(2), [0.1, 0.2])
    assert res["bond_dims"] == [[[2, 4]] * 2, [[2, 3]] * 2, [[2, 2]] * 2]


def test_run_benchmark_compresses_cumulatively_in_place():
    mps = _mps(2)
    B.run_benchmark(mps, _tensors(2), [0.1, 0.3, 0.5])
    assert [m.cuts for m in mps] == [[0.1, 0.3, 0.5]] * 2


def test_run_benchmark_without_cutoffs_measures_once():
    res = B.run_benchmark(_mps(2), _tensors(2), [])
    assert np.asarray(res["ssim"]).shape == (2, 1) and res["bond_dims"] == [[[2, 4]] * 2]


def test_run_benchmark_prints_status(capsys):
    B.run_benchmark(_mps(1), _tensors(1), [0.1, 0.2])
    out = capsys.readouterr().out
    assert "Status: 50.00% - Cutoff: 0.1" in out and "Status: 100.00% - Cutoff: 0.2" in out


def test_run_benchmark_length_mismatch():
    with pytest.raises(IndexError):
        B.run_benchmark(_mps(3), _tensors(2), [0.1])


def test_run_benchmark_empty_list():
    res = B.run_benchmark([], [], [0.1])
    assert all(v == [] for v in res.values())


# ---- load_tensors / run_full_benchmark -------------------------------------------------------------------------
def test_load_tensors_reads_gz_through_nib():
    data, bits = B.load_tensors(["a.nii.gz", "b.nii.gz"], ".gz", shape=(2, 3, 4))
    assert _FakeNib.loaded == ["a.nii.gz", "b.nii.gz"] and bits == [16, 16]
    assert [d.shape for d in data] == [(2, 3, 4)] * 2


def test_load_tensors_rejects_other_endings():
    with pytest.raises(ValueError):
        B.load_tensors(["a.nii"], ".nii")


def _dataset(tmp_path, n=2):
    data = tmp_path / "data"
    data.mkdir()
    for i in range(n):
        np.savez(data / f"clip{i}.npz", sequence=np.arange(60, dtype=np.float32).reshape(3, 4, 5) + i)
    return data


def test_run_full_benchmark_relative_result_goes_under_src_evaluation_results(tmp_path, monkeypatch):
    data = _dataset(tmp_path)
    monkeypatch.chdir(tmp_path)
    B.run_full_benchmark(data, [0.1], "run.json", datatype="Video", mode="Std", ending=".npz")
    res = json.loads((tmp_path / "src/evaluation/results/run.json").read_text())
    assert set(res) == {"datatype", "mode", "files", "cutoff_list", "bitsize_list", "shapes", "ssim", "compression_ratio",
                        "bond_dims", "psnr", "fidelity", "storage", "gzip_bytes", "gzip_ratio"}
    assert res["datatype"] == "Video" and res["mode"] == "Std" and res["cutoff_list"] == [0.1]
    assert res["bitsize_list"] == [32, 32] and res["shapes"] == [[3, 4, 5]] * 2 and len(res["files"]) == 2
    assert np.asarray(res["ssim"]).shape == (2, 2) and all(m.mode == "Std" for m in _FakeNDMPS.created)


def test_run_full_benchmark_keeps_an_already_prefixed_path(tmp_path, monkeypatch):
    data = _dataset(tmp_path)
    monkeypatch.chdir(tmp_path)
    B.run_full_benchmark(data, [0.1], "src/evaluation/results/x.json", ending=".npz")
    assert (tmp_path / "src/evaluation/results/x.json").exists()
    assert not (tmp_path / "src/evaluation/results/src").exists()


def test_run_full_benchmark_keeps_an_absolute_path(tmp_path):
    data = _dataset(tmp_path)
    target = tmp_path / "elsewhere" / "abs.json"
    B.run_full_benchmark(data, [0.1], str(target), ending=".npz")
    assert json.loads(target.read_text())["cutoff_list"] == [0.1]


def test_run_full_benchmark_start_end_and_mri_slices(tmp_path):
    data = _dataset(tmp_path, n=3)
    target = tmp_path / "slices.json"
    B.run_full_benchmark(data, [0.1], str(target), datatype="MRI_Slice", ending=".npz", start=1, end=2)
    res = json.loads(target.read_text())
    assert len(res["files"]) == 1 and res["shapes"] == [[4, 5], [3, 5], [3, 4]] and res["bitsize_list"] == [32] * 3


def test_run_full_benchmark_without_files(tmp_path):
    (tmp_path / "empty").mkdir()
    with pytest.raises(FileNotFoundError):
        B.run_full_benchmark(tmp_path / "empty", [0.1], str(tmp_path / "r.json"), ending=".npz")
    assert not Path(tmp_path / "r.json").exists()
