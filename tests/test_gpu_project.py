"""Maximum / minimum intensity projections (``NDMPS.project``) on the device: parity with numpy's max / min of the full
reconstruction and of the oracle's float64 contraction of the same cores, in Std and DCT mode, float32 and float64,
uncapped and capped, over every axis of every indexed result of the region tests' boxes; bit-exactness against the
region decode when one block covers the box; state after ``compress`` and quantised replace; NaN propagation; errors;
the C ABI's argument checks; and the workspace bound that makes the blocked path worth having."""
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


def check_projections(obj, dtype, with_oracle=True, boxes=None):
    full = obj.to_tensor_device()
    full_np = full.cpu().numpy()
    tol = TOL[dtype] * float(np.abs(full_np).max())
    ref = oracle_of(obj) if with_oracle else None
    for name, index in boxes or _boxes(obj.shape):
        sel = full_np[index]
        for axis in range(-sel.ndim, sel.ndim):
            for op in ("max", "min"):
                if sel.shape[axis] == 0:
                    with pytest.raises(ValueError):
                        obj.project(axis, op, index)
                    continue
                want = getattr(np, op)(sel, axis=axis)
                got_dev = obj.project_device(axis, op, index)
                assert got_dev.is_cuda and got_dev.dtype == full.dtype and got_dev.is_contiguous(), (name, axis, op)
                got = obj.project(axis, op, index)
                assert got.shape == want.shape and got.dtype == want.dtype, (name, axis, op, got.shape, want.shape)
                if want.size == 0:
                    continue
                assert np.abs(got - want).max() <= tol, (name, axis, op, float(np.abs(got - want).max()), tol)
                if ref is not None:
                    r = getattr(np, op)(ref[index], axis=axis)
                    assert np.abs(got.astype(np.float64) - r).max() <= tol, (name, axis, op)


def _whole_axes(shape):
    """the boxes of a large volume: the whole tensor and a 40-slice slab (every axis of each is projected)"""
    return [("full", ()), ("slab", (slice(shape[0] // 4, shape[0] // 4 + 40),))]


@pytest.mark.parametrize("chi", [None, 16], ids=["uncapped", "chi16"])
@pytest.mark.parametrize("mode", ["Std", "DCT"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_projection_matches_full_reconstruction_and_oracle(NDMPS, shape, dtype, mode, chi):
    big = shape == (256, 256, 256)
    obj = build(NDMPS, shape, dtype, mode, chi)
    check_projections(obj, dtype, boxes=_whole_axes(shape) if big else None)


def _one_block_boxes(shape):
    return [b for b in _boxes(shape) if b[0] in ("unaligned", "wrap", "voxel") or b[0].startswith("int")]


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape", [(30, 40, 50), (16, 16, 8, 20), (64, 64, 64)], ids=lambda s: "x".join(map(str, s)))
def test_one_block_equals_the_region_decode_bit_for_bit(NDMPS, shape, dtype):
    """Same T from the same product, and max / min are exact: a box that fits one block projects to exactly numpy's
    max / min of ``contract_region`` on the box."""
    from imgcompressionmps import _native as N
    from imgcompressionmps import _ops
    obj = build(NDMPS, shape, dtype, "Std", None)
    plan = _ops.plan_for(shape)
    for name, index in _one_block_boxes(shape):
        lo, hi, _ = _ops.region_box(shape, index)
        box = _ops.contract_region(obj.mps.cores, shape, lo, hi).cpu().numpy()
        for axis in range(len(shape)):
            info, _, _ = plan.project_debug(lo, hi, axis, (16 << 20) // np.dtype(dtype).itemsize)
            assert info["blocks"] == 1, (name, info)
            for op in ("max", "min"):
                got = _ops.project_region(obj.mps.cores, shape, lo, hi, axis, op).cpu().numpy()
                assert np.array_equal(got, getattr(np, op)(box, axis=axis)), (name, axis, op)
    # the 256^3 volume needs several blocks; the chunk cover itself is checked exactly on the host (test_project.py)
    plan = _ops.plan_for((256, 256, 256))
    assert plan.project_debug([0, 0, 0], [256, 256, 256], 0, (16 << 20) // 4)[0]["blocks"] > 1


@pytest.mark.parametrize("shape,dtype", [((6291456,), np.float32), ((3000000,), np.float64)], ids=["6291456-f32", "3000000-f64"])
def test_multi_block_1d_signal(NDMPS, shape, dtype):
    """A 1-D signal whose decode product needs several blocks along its only axis: every block reduces its own
    positions into the one output value (numpy's max / min exactly, up to the reconstruction's rounding)."""
    from imgcompressionmps import _ops
    info, _, _ = _ops.plan_for(shape).project_debug([0], list(shape), 0, (16 << 20) // np.dtype(dtype).itemsize)
    assert info["blocks"] > 1, info
    obj = NDMPS.from_tensor(smooth(shape, seed=4).astype(dtype))
    check_projections(obj, dtype, with_oracle=False,
                      boxes=[("full", ()), ("tail", (slice(shape[0] // 3, None),)), ("short", (slice(5, 900),))])


@pytest.mark.parametrize("mode", ["Std", "DCT"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape", [(30, 40, 50), (16, 16, 8, 20)], ids=lambda s: "x".join(map(str, s)))
def test_projection_after_compress_and_quantised_replace(NDMPS, shape, dtype, mode):
    obj = NDMPS.from_tensor(smooth(shape, seed=1).astype(dtype), mode=mode)
    before = obj.bond_sizes()
    obj.compress(0.1)
    assert obj.bond_sizes() != before
    check_projections(obj, dtype)
    obj.compress_to_dtype(np.uint16, replace=True)
    check_projections(obj, dtype)


@pytest.mark.parametrize("shape", [(7,), (1, 4), (5, 1, 3)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("mode", ["Std", "DCT"])
def test_single_core_and_extent_one_shapes(NDMPS, shape, mode):
    obj = NDMPS.from_tensor(np.random.default_rng(3).random(shape), mode=mode)
    assert len(obj.mps.cores) == 1
    check_projections(obj, np.float64)
    got = obj.project(0)
    if len(shape) == 1:
        assert got.shape == () and abs(float(got) - obj.to_tensor().max()) <= 1e-12


@pytest.mark.parametrize("mode", ["Std", "DCT"])
def test_nan_propagates_as_in_numpy(NDMPS, mode):
    shape = (30, 40, 50)
    obj = NDMPS.from_tensor(smooth(shape, seed=2), mode=mode)
    cores = [c.clone() for c in obj.mps.cores]
    mid = len(cores) // 2
    cores[mid].view(-1)[cores[mid].numel() // 3] = float("nan")
    obj.replace_tensordata(cores)
    full = obj.to_tensor()
    assert np.isnan(full).any()
    scale = float(np.abs(obj.mps.cores[0].cpu().numpy()).max()) if np.isnan(full).all() else np.nanmax(np.abs(full))
    for index in ((), (slice(3, 20), 7)):
        sel = full[index]
        for axis in range(sel.ndim):
            for op in ("max", "min"):
                got, want = obj.project(axis, op, index), getattr(np, op)(sel, axis=axis)
                assert np.array_equal(np.isnan(got), np.isnan(want)), (index, axis, op)
                ok = ~np.isnan(want)
                assert not ok.any() or np.abs(got[ok] - want[ok]).max() <= 1e-12 * scale, (index, axis, op)


def test_projection_errors_and_unknown_mode(NDMPS):
    obj = build(NDMPS, (30, 40, 50), np.float32, "Std", None)
    for bad in ((3, "max", None), (-4, "max", None), (0, "mean", None), (1, "max", (0, slice(None), 2)),
                (0, "max", (1, 2, 3)), (0, "max", (slice(5, 5),))):
        with pytest.raises(ValueError):
            obj.project(*bad)
    with pytest.raises(IndexError):
        obj.project(0, "max", (30,))
    empty = obj.project_device(0, "min", (slice(None), slice(7, 7)))
    assert empty.is_cuda and tuple(empty.shape) == (0, 50)
    obj.mode = "other"
    try:
        assert obj.project(0) is None and obj.project_device(1, "min", (2,)) is None
        with pytest.raises(ValueError):
            obj.project(0, "sum")
    finally:
        obj.mode = "Std"


def _abi(obj, lo, hi, axis, op, out):
    from imgcompressionmps import _native as N
    from imgcompressionmps import _ops
    cores = obj.mps.cores
    N.check(N.load_library().ndmps_project_region(N.handle(), _ops.plan_for(obj.shape).handle, N.ptr_array(cores),
                                                  N.dtype_code(cores[0].dtype), N.i64_array(_ops._ranks_of(cores)),
                                                  N.i64_array(lo), N.i64_array(hi), int(axis), int(op), 0,
                                                  None if out is None else N.ptr(out)), "ndmps_project_region")


def test_abi_rejects_bad_arguments_and_ignores_an_empty_other_axis(NDMPS):
    obj = build(NDMPS, (12, 18, 10), np.float64, "Std", None)
    out = torch.empty(18 * 10, dtype=torch.float64, device="cuda")
    full = [0, 0, 0], [12, 18, 10]
    for lo, hi, axis, op in [(*full, 3, 1), (*full, -1, 1), (*full, 0, 0), (*full, 0, 3), ([0, 0, 0], [13, 18, 10], 0, 1),
                             ([4, 0, 0], [4, 18, 10], 0, 1)]:
        with pytest.raises(ValueError):
            _abi(obj, lo, hi, axis, op, out)
    _abi(obj, [0, 5, 0], [12, 5, 10], 0, 1, None)                 # empty on axis 1: a no-op, out may be NULL
    _abi(obj, *full, 0, 1, out)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy().reshape(18, 10), obj.project(0))


def test_projection_workspace_is_bounded_by_one_block(NDMPS):
    """A MIP along each axis of a 256^3 float32 MPS at chi = 128, in a fresh thread (its own context and arena): the
    arena's high-water mark stays under 24 MB, 3/8 of the 64 MB tensor (the full reconstruction needs the tensor
    twice), and torch allocates nothing but the 256 KB result."""
    from imgcompressionmps import _native as N
    shape = (256, 256, 256)
    obj = NDMPS.from_tensor(smooth(shape, seed=5).astype(np.float32), max_bond=128)
    full = obj.to_tensor_device()
    want = [full.amax(dim=a).cpu().numpy() for a in range(3)]
    scale = float(full.abs().max())
    del full
    torch.cuda.synchronize()
    result = {}

    def run():
        try:
            got, peaks = [], []
            for a in range(3):
                torch.cuda.synchronize()
                torch.cuda.reset_peak_memory_stats()
                base = torch.cuda.memory_allocated()
                out = obj.project_device(a)
                torch.cuda.synchronize()
                peaks.append(torch.cuda.max_memory_allocated() - base)
                got.append(out.cpu().numpy())
            obj.project_device(0, index=(slice(0, 1), 0, slice(0, 2)))    # the high-water mark folds in at the next reset
            torch.cuda.synchronize()
            result.update(got=got, peaks=peaks, ws=N.context().stat("workspace_bytes"))
        except Exception as exc:                            # surfaced in the main thread
            result["error"] = exc

    t = threading.Thread(target=run)
    t.start()
    t.join()
    if "error" in result:
        raise result["error"]
    tensor_bytes = 4 * 256 ** 3
    assert 0 < result["ws"] < 3 * tensor_bytes / 8, result["ws"]
    for a in range(3):
        assert result["peaks"][a] <= 4 * 256 * 256, (a, result["peaks"])
        assert np.abs(result["got"][a] - want[a]).max() <= 1e-5 * scale, a
