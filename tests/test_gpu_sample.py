"""Interpolated sampling (``NDMPS.sample``, ``sample_grid``, ``sample_grid_device``) on the device: parity with
``scipy.ndimage.map_coordinates(order=1, mode="nearest")`` on the full reconstruction and on the oracle's float64
contraction of the same cores, in Std and DCT mode, float32 and float64, uncapped and capped, after ``compress`` and
``compress_to_dtype(replace=True)``; affine grids against the same grid built in numpy; input forms; errors; and the
workspace bound of an oblique plane."""
import threading

import numpy as np
import pytest
from scipy.ndimage import map_coordinates

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from test_gpu_region import SHAPES, TOL, build, oracle_of, smooth   # noqa: E402


@pytest.fixture(scope="module")
def NDMPS():
    from imgcompressionmps.core.ndmps import NDMPS
    return NDMPS


def interp(vol, coords):
    return map_coordinates(vol, np.asarray(coords, dtype=np.float64).T, order=1, mode="nearest")


def coords_for(shape, seed=0, k=600):
    """Random points in [-2, extent + 1] plus exact integers, the upper edge extent - 1, fractions 0 and just below 1,
    negatives and duplicates."""
    rng = np.random.default_rng(seed)
    ext = np.array(shape, dtype=np.float64)
    rand = rng.uniform(-2.0, ext + 1.0, size=(k, len(shape)))
    ints = np.stack([rng.integers(0, n, size=40) for n in shape], axis=1).astype(np.float64)
    below_one = np.nextafter(ints + 1.0, -np.inf)          # i + (1 - ulp): the largest fraction below the next voxel
    first = np.full((1, len(shape)), 1.0 - 2.0 ** -52)
    edge = np.vstack([ext - 1, np.zeros(len(shape)), np.nextafter(ext - 1, -np.inf)])
    neg = -np.abs(rand[:20])
    dup = np.repeat(rand[:5], 3, axis=0)
    return np.vstack([rand, ints, below_one, first, edge, neg, dup])


def check_sample(obj, dtype, with_oracle=True, seed=0):
    full = obj.to_tensor()
    tol = TOL[dtype] * float(np.abs(full).max())
    coords = coords_for(obj.shape, seed)
    got = obj.sample(coords)
    assert isinstance(got, np.ndarray) and got.dtype == full.dtype and got.shape == (len(coords),)
    want = interp(full.astype(np.float64), coords)
    assert np.abs(got - want).max() <= tol, (float(np.abs(got - want).max()), tol)
    if with_oracle:
        ref = interp(oracle_of(obj), coords)
        assert np.abs(got - ref).max() <= tol, (float(np.abs(got - ref).max()), tol)


@pytest.mark.parametrize("chi", [None, 16], ids=["uncapped", "chi16"])
@pytest.mark.parametrize("mode", ["Std", "DCT"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_sample_matches_map_coordinates_and_oracle(NDMPS, shape, dtype, mode, chi):
    check_sample(build(NDMPS, shape, dtype, mode, chi), dtype)


@pytest.mark.parametrize("mode", ["Std", "DCT"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape", [(30, 40, 50), (16, 16, 8, 20), (64, 64, 64)], ids=lambda s: "x".join(map(str, s)))
def test_sample_after_compress_and_quantised_replace(NDMPS, shape, dtype, mode):
    obj = NDMPS.from_tensor(smooth(shape, seed=1).astype(dtype), mode=mode)
    before = obj.bond_sizes()
    obj.compress(0.1)
    assert obj.bond_sizes() != before
    check_sample(obj, dtype, seed=1)
    obj.compress_to_dtype(np.uint16, replace=True)
    check_sample(obj, dtype, seed=2)


@pytest.mark.parametrize("mode", ["Std", "DCT"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape", [(8, 9), (30, 40, 50), (16, 16, 8, 20)], ids=lambda s: "x".join(map(str, s)))
def test_sample_at_integers_equals_values_at(NDMPS, shape, dtype, mode):
    obj = build(NDMPS, shape, dtype, mode, None)
    full = obj.to_tensor()
    rng = np.random.default_rng(5)
    pts = np.stack([rng.integers(0, n, size=300) for n in shape], axis=1)
    got = obj.sample(pts)
    assert got.dtype == full.dtype
    assert np.array_equal(got, obj.values_at(pts))        # one kernel: the same arithmetic for an integer point


@pytest.mark.parametrize("shape", [(7,), (1, 4), (5, 1, 3), (16, 1, 20), (1, 30, 40), (12, 18, 1)],
                         ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("mode", ["Std", "DCT"])
def test_single_core_and_extent_one_axes(NDMPS, shape, mode):
    """An extent-1 axis has no factors to split, so these are all single-core MPS (L = 1: X is the core, no W^T)."""
    x = np.random.default_rng(3).random(shape)
    obj = NDMPS.from_tensor(x, mode=mode)
    assert len(obj.mps.cores) == 1
    check_sample(obj, np.float64)


def grid_coords(origin, steps, shape):
    idx = np.stack(np.meshgrid(*[np.arange(n, dtype=np.float64) for n in shape], indexing="ij"), axis=-1)
    return (np.asarray(origin, dtype=np.float64) + idx @ np.asarray(steps, dtype=np.float64)).reshape(-1, len(origin))


def _grids():
    u = np.array([1.0, 1.0, 0.0]) / np.sqrt(2.0)
    v = np.array([1.0, -1.0, 1.0]) / np.sqrt(3.0)
    c = np.array([14.5, 19.5, 24.5])
    return [
        ("oblique plane", (30, 40, 50), c - 20.0 * (u + v), [u * 0.9, v * 1.1], (41, 37)),
        ("line", (30, 40, 50), [-1.5, 3.25, 60.0], [[0.37, 0.41, -0.83]], (90,)),
        ("resample", (30, 40, 50), [0.0, 0.0, 0.0], np.diag([29 / 16, 39 / 22, 49 / 60]), (17, 23, 61)),
        ("4-D", (16, 16, 8, 20), [0.3, -0.2, 1.1, 2.0], np.diag([0.7, 1.3, 0.6, 1.7]) + 0.05, (9, 13, 5, 11)),
    ]


@pytest.mark.parametrize("mode", ["Std", "DCT"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("case", _grids(), ids=lambda c: c[0])
def test_grid_equals_sample_of_the_same_grid(NDMPS, case, dtype, mode):
    _, shape, origin, steps, out_shape = case
    obj = build(NDMPS, shape, dtype, mode, None)
    full = obj.to_tensor()
    tol = TOL[dtype] * float(np.abs(full).max())
    got = obj.sample_grid(origin, steps, out_shape)
    assert isinstance(got, np.ndarray) and got.shape == out_shape and got.dtype == full.dtype
    coords = grid_coords(origin, steps, out_shape)
    assert np.abs(got.reshape(-1) - obj.sample(coords)).max() <= tol
    assert np.abs(got.reshape(-1) - interp(full.astype(np.float64), coords)).max() <= tol
    dev = obj.sample_grid_device(origin, steps, out_shape)
    assert dev.is_cuda and tuple(dev.shape) == out_shape
    assert np.array_equal(dev.cpu().numpy(), got)


def test_zero_extent_grid(NDMPS):
    obj = build(NDMPS, (30, 40, 50), np.float32, "Std", None)
    got = obj.sample_grid([0, 0, 0], [[1, 0, 0], [0, 1, 0]], (0, 5))
    assert isinstance(got, np.ndarray) and got.shape == (0, 5) and got.dtype == np.float32
    dev = obj.sample_grid_device([0, 0, 0], np.eye(3), (4, 0, 2))
    assert dev.is_cuda and tuple(dev.shape) == (4, 0, 2)


def test_input_forms(NDMPS):
    obj = build(NDMPS, (30, 40, 50), np.float64, "Std", None)
    full = obj.to_tensor()
    tol = 1e-12 * float(np.abs(full).max())
    coords = coords_for(obj.shape, seed=7, k=200)
    want = interp(full, coords)
    got_dev = obj.sample(torch.as_tensor(coords, device="cuda"))
    assert got_dev.is_cuda and got_dev.shape == (len(coords),) and got_dev.dtype == torch.float64
    assert np.abs(got_dev.cpu().numpy() - want).max() <= tol
    c32 = coords.astype(np.float32)
    want32 = interp(full, c32.astype(np.float64))
    assert np.abs(obj.sample(c32) - want32).max() <= tol
    assert np.abs(obj.sample(torch.as_tensor(c32, device="cuda")).cpu().numpy() - want32).max() <= tol
    ints = np.stack([np.arange(-3, 60) % 33, np.arange(63) % 41, np.arange(63) - 5], axis=1)   # some clamp
    want_i = interp(full, ints)
    for form in (ints, ints.astype(np.int32), ints.astype(np.int16), torch.as_tensor(ints, device="cuda")):
        got = obj.sample(form)
        got = got.cpu().numpy() if isinstance(got, torch.Tensor) else got
        assert np.abs(got - want_i).max() <= tol
    assert obj.sample(np.zeros((0, 3))).shape == (0,)
    empty = obj.sample(torch.zeros((0, 3), device="cuda"))
    assert empty.is_cuda and empty.shape == (0,)


def test_sample_errors(NDMPS):
    obj = build(NDMPS, (30, 40, 50), np.float32, "Std", None)
    bad = [np.zeros((4, 2)), np.zeros(3), np.zeros((2, 4)), np.zeros((2, 3, 1)), torch.zeros((3, 2), device="cuda"),
           torch.zeros((1, 3)),                                                  # a CPU tensor
           np.zeros((2, 3), dtype=bool), np.zeros((2, 3), dtype=np.complex128), torch.zeros((2, 3), dtype=torch.bool,
                                                                                            device="cuda"),
           np.array([[0.0, np.nan, 1.0]]), np.array([[np.inf, 0.0, 1.0]]), np.array([[0.0, 1.0, -np.inf]]),
           torch.tensor([[0.0, float("nan"), 1.0]], device="cuda"), torch.tensor([[0.0, 1.0, float("inf")]], device="cuda")]
    for b in bad:
        with pytest.raises(ValueError):
            obj.sample(b)
    ok_origin, ok_steps = [0.0, 0.0, 0.0], [[1.0, 0.0, 0.0]]
    for origin, steps, shape in [([0.0, 0.0], ok_steps, (4,)),                          # origin length
                                 (ok_origin, [[1.0, 0.0]], (4,)),                          # steps width
                                 (ok_origin, np.zeros((0, 3)), ()),                        # m = 0
                                 (ok_origin, np.zeros((9, 3)), (1,) * 9),                  # m = 9
                                 (ok_origin, [1.0, 0.0, 0.0], (4,)),                       # steps not 2-D
                                 (ok_origin, ok_steps, (4, 4)),                            # shape length
                                 (ok_origin, ok_steps, (-1,)),                             # negative extent
                                 ([np.nan, 0.0, 0.0], ok_steps, (4,)),
                                 (ok_origin, [[np.inf, 0.0, 0.0]], (4,)),
                                 (ok_origin, [[1e308, 0.0, 0.0]], (4,)),                   # overflows to inf
                                 ([True, False, True], ok_steps, (4,)),
                                 (ok_origin, [[1j, 0, 0]], (4,))]:
        with pytest.raises(ValueError):
            obj.sample_grid(origin, steps, shape)
        with pytest.raises(ValueError):
            obj.sample_grid_device(origin, steps, shape)
    with pytest.raises(TypeError):
        obj.sample_grid(ok_origin, ok_steps, (2.5,))


def test_unknown_mode_returns_none_after_the_checks(NDMPS):
    obj = NDMPS.from_tensor(smooth((12, 18, 10)))
    obj.mode = "other"
    assert obj.sample(np.zeros((3, 3))) is None
    assert obj.sample_grid([0, 0, 0], np.eye(3), (2, 2, 2)) is None
    assert obj.sample_grid_device([0, 0, 0], np.eye(3), (2, 2, 2)) is None
    with pytest.raises(ValueError):
        obj.sample(np.array([[np.nan, 0, 0]]))
    with pytest.raises(ValueError):
        obj.sample_grid([0, 0], np.eye(3), (2, 2, 2))


def test_kernel_writes_nan_for_a_non_finite_coordinate(NDMPS):
    """The Python layer refuses such coordinates; passed straight to the kernel, they give NaN and read no core."""
    from imgcompressionmps import _ops
    obj = build(NDMPS, (30, 40, 50), np.float64, "Std", None)
    coords = torch.tensor([[0.5, 0.0, 0.0], [float("nan"), 1.0, 1.0], [2.0, float("inf"), 3.0], [1.0, 2.0, -float("inf")],
                           [29.0, 39.0, 49.0]], dtype=torch.float64, device="cuda")
    got = _ops.sample_points(obj.mps.cores, obj.shape, coords).cpu().numpy()
    full = obj.to_tensor()
    assert np.isnan(got[1:4]).all()
    want = interp(full, coords.cpu().numpy()[[0, 4]])
    assert np.abs(got[[0, 4]] - want).max() <= 1e-12 * float(np.abs(full).max())


def _abi(obj, fn, **kw):
    from imgcompressionmps import _native as N
    from imgcompressionmps import _ops
    import ctypes as C
    cores = obj.mps.cores
    lib = N.load_library()
    a = dict(ctx=N.handle(), plan=_ops.plan_for(obj.shape).handle, cores=N.ptr_array(cores),
             dtype=N.dtype_code(cores[0].dtype), ranks=N.i64_array(_ops._ranks_of(cores)),
             out=N.ptr(torch.empty(64, dtype=cores[0].dtype, device="cuda")), idct=0)
    a.update(kw)
    if fn == "points":
        coords = a.get("coords", N.ptr(torch.zeros((4, 3), dtype=torch.float64, device="cuda")))
        rc = lib.ndmps_sample_points(a["ctx"], a["plan"], a["cores"], a["dtype"], a["ranks"], coords, a.get("count", 4),
                                     a["idct"], a["out"])
    else:
        origin = a.get("origin", [0.0, 0.0, 0.0])
        origin = None if origin is None else np.ascontiguousarray(origin, dtype=np.float64)
        steps = np.ascontiguousarray(a.get("steps", [[1.0, 0.0, 0.0]]), dtype=np.float64)
        shape = a.get("shape", [4])
        rc = lib.ndmps_sample_grid(a["ctx"], a["plan"], a["cores"], a["dtype"], a["ranks"],
                                   None if origin is None else origin.ctypes.data_as(N.p_f64),
                                   steps.ctypes.data_as(N.p_f64), N.i64_array(shape), a.get("m", len(shape)), a["idct"],
                                   a["out"])
    N.check(rc, "sample abi")
    torch.cuda.synchronize()


def test_abi_rejects_null_and_bad_arguments(NDMPS):
    obj = build(NDMPS, (30, 40, 50), np.float64, "Std", None)
    _abi(obj, "points")
    _abi(obj, "grid")
    for fn, kw in [("points", dict(ctx=None)), ("points", dict(cores=None)), ("points", dict(coords=None)),
                   ("points", dict(out=None)), ("points", dict(count=-1)), ("points", dict(dtype=7)),
                   ("points", dict(ranks=None)),
                   ("grid", dict(plan=None)), ("grid", dict(origin=None)), ("grid", dict(out=None)),
                   ("grid", dict(m=0)), ("grid", dict(m=9, shape=[1] * 9, steps=np.zeros((9, 3)))),
                   ("grid", dict(shape=[-1])), ("grid", dict(origin=[np.nan, 0.0, 0.0])),
                   ("grid", dict(steps=[[np.inf, 0.0, 0.0]])), ("grid", dict(dtype=-1))]:
        with pytest.raises(ValueError):
            _abi(obj, fn, **kw)
    _abi(obj, "points", count=0, coords=None, out=None)           # count 0 writes nothing
    _abi(obj, "grid", shape=[0], out=None)                         # so does a zero extent


def test_oblique_plane_workspace_is_bounded(NDMPS):
    """A 256 x 256 oblique plane of a 256^3 float32 MPS at chi = 128, sampled in a fresh thread (its own context and
    workspace arena), keeps the arena's high-water mark and the torch allocation below 1/8 of the 64 MB tensor."""
    from imgcompressionmps import _native as N
    shape = (256, 256, 256)
    obj = NDMPS.from_tensor(smooth(shape, seed=5).astype(np.float32), max_bond=128)
    u = np.array([1.0, 1.0, 0.0]) / np.sqrt(2.0)
    v = np.array([1.0, -1.0, 1.0]) / np.sqrt(3.0)
    origin = np.full(3, 127.5) - 127.5 * (u + v)
    steps = np.stack([u, v])
    want = interp(obj.to_tensor().astype(np.float64), grid_coords(origin, steps, (256, 256))).reshape(256, 256)
    torch.cuda.synchronize()
    result = {}

    def run():
        try:
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            plane = obj.sample_grid_device(origin, steps, (256, 256))
            torch.cuda.synchronize()
            result["torch"] = torch.cuda.max_memory_allocated() - base
            obj.sample(np.zeros((1, 3)))                   # the high-water mark folds in at the next reset
            torch.cuda.synchronize()
            result["plane"] = plane.cpu().numpy()
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
    assert 0 < result["torch"] < tensor_bytes / 8, result["torch"]
    assert np.abs(result["plane"] - want).max() <= 1e-5 * float(np.abs(want).max())
