"""Box decode (``NDMPS.to_tensor_region``) and point evaluation (``NDMPS.values_at``) on the device: parity with
the full reconstruction and with the oracle's float64 contraction of the same cores, in Std and DCT mode, float32
and float64, uncapped and capped, after ``compress`` and ``compress_to_dtype(replace=True)``; errors; and the
workspace bound that makes the region path worth having."""
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from oracle.ndmps import OracleNDMPS                      # noqa: E402
from test_region import _boxes                            # noqa: E402

SHAPES = [(8, 9), (30, 40, 50), (12, 18, 10), (16, 16, 8, 20), (64, 64, 64), (256, 256, 256)]
TOL = {np.float64: 1e-12, np.float32: 1e-5}


@pytest.fixture(scope="module")
def NDMPS():
    from imgcompressionmps.core.ndmps import NDMPS
    return NDMPS


def smooth(shape, seed=0):
    """A smooth field of modest TT rank (an uncapped sweep of 256^3 stays small) that is not separable."""
    rng = np.random.default_rng(seed)
    g = np.meshgrid(*[np.linspace(-1, 1, n) for n in shape], indexing="ij")
    c = rng.uniform(-0.3, 0.3, size=len(shape))
    r2 = sum((1.0 + 0.5 * a) * (x - ca) ** 2 for a, (x, ca) in enumerate(zip(g, c)))
    if len(shape) > 1:
        r2 = r2 + 0.8 * g[0] * g[1]                           # not a product of per-axis factors
    wave = np.cos(sum((2.0 + a) * x for a, x in enumerate(g)))
    return np.exp(-3.0 * r2) + 0.3 * wave + 0.1 * np.prod([x + 0.5 * a for a, x in enumerate(g)], axis=0)


_CACHE = {}


def build(NDMPS, shape, dtype, mode, chi):
    key = (shape, dtype, mode, chi)
    if key not in _CACHE:
        obj = NDMPS.from_tensor(smooth(shape).astype(dtype), mode=mode, max_bond=chi)
        _CACHE.clear()                                    # keep one object (and its 256^3 reconstruction) alive
        _CACHE[key] = obj
    return _CACHE[key]


def oracle_of(obj):
    """The oracle's float64 to_tensor on the device's own cores (same MPS, reference arithmetic)."""
    cores = [c.detach().cpu().numpy().astype(np.float64) for c in obj.mps.cores]
    return OracleNDMPS(cores, np.array(obj.mps.site_dims), obj.shape, False, None, obj.mode, None).to_tensor()


def check_boxes(obj, dtype, with_oracle=True):
    full = obj.to_tensor_device()
    full_np = full.cpu().numpy()
    scale = float(np.abs(full_np).max())
    tol = TOL[dtype] * scale
    ref = oracle_of(obj) if with_oracle else None
    for name, index in _boxes(obj.shape):
        got_dev = obj.to_tensor_region_device(index)
        assert got_dev.is_cuda and got_dev.dtype == full.dtype and got_dev.is_contiguous(), name
        got = obj.to_tensor_region(index)
        want = full_np[index]
        assert got.shape == want.shape and got.dtype == want.dtype, (name, got.shape, want.shape)
        if want.size == 0:
            continue
        assert np.abs(got - want).max() <= tol, (name, float(np.abs(got - want).max()), tol)
        if ref is not None:
            assert np.abs(got.astype(np.float64) - ref[index]).max() <= tol, (name, float(np.abs(got - ref[index]).max()), tol)


@pytest.mark.parametrize("chi", [None, 16], ids=["uncapped", "chi16"])
@pytest.mark.parametrize("mode", ["Std", "DCT"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_region_matches_full_reconstruction_and_oracle(NDMPS, shape, dtype, mode, chi):
    check_boxes(build(NDMPS, shape, dtype, mode, chi), dtype)


@pytest.mark.parametrize("mode", ["Std", "DCT"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape", [(30, 40, 50), (16, 16, 8, 20), (64, 64, 64)], ids=lambda s: "x".join(map(str, s)))
def test_region_after_compress_and_quantised_replace(NDMPS, shape, dtype, mode):
    obj = NDMPS.from_tensor(smooth(shape, seed=1).astype(dtype), mode=mode)
    before = obj.bond_sizes()
    obj.compress(0.1)
    assert obj.bond_sizes() != before                     # the bonds really changed
    check_boxes(obj, dtype)
    obj.compress_to_dtype(np.uint16, replace=True)
    check_boxes(obj, dtype)


@pytest.mark.parametrize("shape", [(7,), (1, 4), (5, 1, 3)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("mode", ["Std", "DCT"])
def test_single_core_shapes(NDMPS, shape, mode):
    x = np.random.default_rng(3).random(shape)
    obj = NDMPS.from_tensor(x, mode=mode)
    assert len(obj.mps.cores) == 1
    check_boxes(obj, np.float64)
    full = obj.to_tensor()
    coords = np.array(list(np.ndindex(*shape)) * 2, dtype=np.int64)
    got = obj.values_at(coords)
    assert np.abs(got - full[tuple(coords.T)]).max() <= 1e-12 * np.abs(full).max()


@pytest.mark.parametrize("mode", ["Std", "DCT"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape,chi", [((30, 40, 50), None), ((64, 64, 64), 16), ((16, 16, 8, 20), None), ((8, 9), None)],
                         ids=["30x40x50", "64^3-chi16", "16x16x8x20", "8x9"])
def test_values_at(NDMPS, shape, chi, dtype, mode):
    obj = build(NDMPS, shape, dtype, mode, chi)
    full = obj.to_tensor()
    tol = TOL[dtype] * float(np.abs(full).max())
    rng = np.random.default_rng(11)
    pts = np.stack([rng.integers(0, n, size=500) for n in shape], axis=1)
    corners = np.array(list(np.ndindex(*[2] * len(shape)))) * (np.array(shape) - 1)
    dup = np.repeat(pts[:3], 4, axis=0)
    neg = pts[:20] - np.array(shape)                      # negative coordinates count from the end
    for coords in (pts, corners, dup, neg, pts.astype(np.int32)):
        got = obj.values_at(coords)
        assert isinstance(got, np.ndarray) and got.dtype == full.dtype and got.shape == (len(coords),)
        assert np.abs(got - full[tuple(coords.T)]).max() <= tol
        got_dev = obj.values_at(torch.as_tensor(coords, device="cuda"))
        assert got_dev.is_cuda and got_dev.shape == (len(coords),)
        assert np.array_equal(got_dev.cpu().numpy(), got)
    empty = obj.values_at(np.zeros((0, len(shape)), dtype=np.int64))
    assert isinstance(empty, np.ndarray) and empty.shape == (0,)
    empty_dev = obj.values_at(torch.zeros((0, len(shape)), dtype=torch.int64, device="cuda"))
    assert empty_dev.is_cuda and empty_dev.shape == (0,)


def test_values_at_and_region_errors(NDMPS):
    obj = build(NDMPS, (30, 40, 50), np.float32, "Std", None)
    for bad in (np.array([[30, 0, 0]]), np.array([[0, -41, 0]]), torch.tensor([[0, 0, 50]], device="cuda")):
        with pytest.raises(IndexError):
            obj.values_at(bad)
    for bad in (np.zeros((4, 2), dtype=np.int64), np.zeros(3, dtype=np.int64), np.zeros((2, 4), dtype=np.int64),
                torch.zeros((3, 2), dtype=torch.int64, device="cuda"), torch.zeros((1, 3), dtype=torch.int64)):
        with pytest.raises(ValueError):
            obj.values_at(bad)
    with pytest.raises(IndexError):
        obj.values_at(np.zeros((2, 3), dtype=np.float64))
    with pytest.raises(IndexError):
        obj.to_tensor_region((30,))
    with pytest.raises(IndexError):
        obj.to_tensor_region((0, 0, 0, 0))
    with pytest.raises(ValueError):
        obj.to_tensor_region((slice(None, None, 2),))


def test_unknown_mode_returns_none(NDMPS):
    obj = NDMPS.from_tensor(smooth((12, 18, 10)))
    obj.mode = "other"
    assert obj.to_tensor() is None
    assert obj.to_tensor_region((1,)) is None and obj.to_tensor_region_device((slice(2, 5),)) is None
    assert obj.values_at(np.zeros((3, 3), dtype=np.int64)) is None


def test_kernel_writes_nan_for_a_coordinate_outside_the_volume(NDMPS):
    """The Python layer refuses such coordinates; called directly, the kernel reads no core out of bounds and gives NaN."""
    from imgcompressionmps import _ops
    obj = build(NDMPS, (30, 40, 50), np.float64, "Std", None)
    coords = torch.tensor([[0, 0, 0], [30, 0, 0], [0, 0, -51], [29, 39, 49]], dtype=torch.int64, device="cuda")
    got = _ops.evaluate_points(obj.mps.cores, obj.shape, coords).cpu().numpy()
    full = obj.to_tensor()
    assert np.isnan(got[1]) and np.isnan(got[2])
    assert abs(got[0] - full[0, 0, 0]) <= 1e-12 and abs(got[3] - full[29, 39, 49]) <= 1e-12


def test_region_abi_rejects_a_bad_box_and_ignores_an_empty_one(NDMPS):
    from imgcompressionmps import _ops
    obj = build(NDMPS, (12, 18, 10), np.float64, "Std", None)
    for lo, hi in [([0, 0, 0], [13, 18, 10]), ([-1, 0, 0], [2, 2, 2]), ([5, 0, 0], [4, 18, 10])]:
        with pytest.raises(ValueError):
            _abi_region(obj, lo, hi)
    assert _ops.contract_region(obj.mps.cores, obj.shape, [3, 0, 0], [3, 18, 10]).shape == (0, 18, 10)


def _abi_region(obj, lo, hi):
    from imgcompressionmps import _native as N
    from imgcompressionmps import _ops
    cores = obj.mps.cores
    out = torch.empty(1, dtype=cores[0].dtype, device="cuda")
    N.check(N.load_library().ndmps_contract_region(N.handle(), _ops.plan_for(obj.shape).handle, N.ptr_array(cores),
                                                   N.dtype_code(cores[0].dtype), N.i64_array(_ops._ranks_of(cores)),
                                                   N.i64_array(lo), N.i64_array(hi), N.ptr(out)), "ndmps_contract_region")


def test_region_workspace_is_bounded_by_the_box(NDMPS):
    """A 1 x 256 x 256 slice of a 256^3 float32 MPS at chi = 128, decoded in a fresh thread (its own context and
    workspace arena), keeps the arena's high-water mark below 1/8 of the 64 MB tensor; the full reconstruction would
    need the whole tensor twice."""
    from imgcompressionmps import _native as N
    shape = (256, 256, 256)
    obj = NDMPS.from_tensor(smooth(shape, seed=5).astype(np.float32), max_bond=128)
    full = obj.to_tensor_device()[100].cpu().numpy()
    result = {}

    def run():
        try:
            sl = obj.to_tensor_region_device((100,))
            obj.to_tensor_region_device((0, 0, slice(0, 2)))   # the high-water mark folds in at the next reset
            torch.cuda.synchronize()
            result["slice"] = sl.cpu().numpy()
            result["ws"] = N.context().stat("workspace_bytes")
        except Exception as exc:                            # surfaced in the main thread
            result["error"] = exc

    t = threading.Thread(target=run)
    t.start()
    t.join()
    if "error" in result:
        raise result["error"]
    tensor_bytes = 4 * 256 ** 3
    assert 0 < result["ws"] < tensor_bytes / 8, result["ws"]
    assert np.abs(result["slice"] - full).max() <= 1e-5 * float(np.abs(full).max())
