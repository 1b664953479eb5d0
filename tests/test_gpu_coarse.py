"""Block-mean decode (``NDMPS.to_tensor_coarse``) on the device: parity with the block mean of the full
reconstruction and of the oracle's float64 contraction of the same cores, in Std and DCT mode, float32 and float64,
uncapped and capped, for every box of the coarse shape; after ``compress`` and ``compress_to_dtype(replace=True)``;
errors of the public methods and of ``ndmps_marginalize``; the block-averaged inverse DCT against scipy; and the
memory bound that makes the coarse path worth having."""
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from test_coarse import block_mean, level_cases           # noqa: E402
from test_gpu_region import SHAPES, TOL, build, oracle_of, smooth   # noqa: E402
from test_region import _boxes                            # noqa: E402


@pytest.fixture(scope="module")
def NDMPS():
    from imgcompressionmps.core.ndmps import NDMPS
    return NDMPS


def check_coarse(obj, dtype, with_oracle=True):
    full = obj.to_tensor_device().cpu().numpy()
    scale = float(np.abs(full).max())
    tol = TOL[dtype] * scale
    ref = oracle_of(obj) if with_oracle else None
    for levels in level_cases(obj.shape):
        cshape = obj.coarse_shape(levels)
        block = tuple(s // c for s, c in zip(obj.shape, cshape))
        want_all = block_mean(full.astype(np.float64), block)
        ref_all = block_mean(ref, block) if ref is not None else None
        for name, index in [("none", None)] + _boxes(cshape):
            got_dev = obj.to_tensor_coarse_device(levels, index)
            assert got_dev.is_cuda and got_dev.dtype == obj.mps.cores[0].dtype and got_dev.is_contiguous(), name
            got = obj.to_tensor_coarse(levels, index)
            want = want_all if index is None else want_all[index]
            assert got.shape == want.shape and got.dtype == full.dtype, (levels, name, got.shape, want.shape)
            if want.size == 0:
                continue
            err = float(np.abs(got - want).max())
            assert err <= tol, (levels, name, err, tol)
            if ref_all is not None:
                r = ref_all if index is None else ref_all[index]
                err = float(np.abs(got.astype(np.float64) - r).max())
                assert err <= tol, (levels, name, "oracle", err, tol)
    # levels 0 is the reconstruction itself
    assert np.abs(obj.to_tensor_coarse(0) - full).max() <= tol
    mid = tuple(n // 2 for n in obj.shape[:-1])
    assert np.abs(obj.to_tensor_coarse(0, mid) - obj.to_tensor_region(mid)).max() <= tol


@pytest.mark.parametrize("chi", [None, 16], ids=["uncapped", "chi16"])
@pytest.mark.parametrize("mode", ["Std", "DCT"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_coarse_matches_block_mean_of_full_reconstruction_and_oracle(NDMPS, shape, dtype, mode, chi):
    check_coarse(build(NDMPS, shape, dtype, mode, chi), dtype)


@pytest.mark.parametrize("mode", ["Std", "DCT"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape", [(30, 40, 50), (16, 16, 8, 20)], ids=lambda s: "x".join(map(str, s)))
def test_coarse_after_compress_and_quantised_replace(NDMPS, shape, dtype, mode):
    obj = NDMPS.from_tensor(smooth(shape, seed=1).astype(dtype), mode=mode)
    before = obj.bond_sizes()
    obj.compress(0.1)
    assert obj.bond_sizes() != before
    check_coarse(obj, dtype)
    obj.compress_to_dtype(np.uint16, replace=True)
    check_coarse(obj, dtype)


@pytest.mark.parametrize("shape", [(7,), (1, 4)], ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("mode", ["Std", "DCT"])
def test_coarse_single_core_shapes(NDMPS, shape, mode):
    obj = NDMPS.from_tensor(np.random.default_rng(3).random(shape), mode=mode)
    assert len(obj.mps.cores) == 1
    check_coarse(obj, np.float64)


def test_coarse_argument_errors_and_unknown_mode(NDMPS):
    obj = build(NDMPS, (30, 40, 50), np.float32, "Std", None)
    for bad in (True, 1.0, [1, 1.0, 0]):
        with pytest.raises(TypeError):
            obj.to_tensor_coarse(bad)
    for bad in (-1, 99, [1, 1]):
        with pytest.raises(ValueError):
            obj.to_tensor_coarse_device(bad)
    with pytest.raises(IndexError):
        obj.to_tensor_coarse(1, (6,))                    # coarse shape (6, 20, 10)
    with pytest.raises(IndexError):
        obj.to_tensor_coarse(1, (0, 0, 0, 0))
    with pytest.raises(ValueError):
        obj.to_tensor_coarse(1, (slice(None, None, 2),))
    other = NDMPS.from_tensor(smooth((12, 18, 10)))
    other.mode = "other"
    assert other.to_tensor_coarse(1) is None and other.to_tensor_coarse_device(1, (slice(0, 2),)) is None
    with pytest.raises(ValueError):
        other.to_tensor_coarse(-1)


def _abi_marginalize(obj, drop, caps):
    from imgcompressionmps import _native as N
    from imgcompressionmps import _ops
    cores = obj.mps.cores
    outs = [torch.empty(max(int(c), 1), dtype=cores[0].dtype, device="cuda") for c in caps]
    N.check(N.load_library().ndmps_marginalize(N.handle(), _ops.plan_for(obj.shape).handle, N.ptr_array(cores),
                                               N.dtype_code(cores[0].dtype), N.i64_array(_ops._ranks_of(cores)),
                                               N.i64_array(drop), N.ptr_array(outs), N.i64_array(caps)),
            "ndmps_marginalize")


def test_marginalize_abi_rejects_bad_levels_and_small_capacity(NDMPS):
    from imgcompressionmps import _native as N
    from imgcompressionmps import _ops
    obj = build(NDMPS, (30, 40, 50), np.float64, "Std", None)
    L = len(obj.mps.cores)
    for drop in ([-1, 0, 0], [0, L + 1, 0]):
        with pytest.raises(ValueError):
            _abi_marginalize(obj, drop, [1 << 20] * L)
    plan = _ops.coarse_plan(obj.shape, 1)
    red = _ops.marginalize(obj.mps.cores, obj.shape, 1)
    caps = [c.numel() for c in red]
    caps[plan.levels // 2] -= 1
    with pytest.raises(N.NativeError):
        _abi_marginalize(obj, [1, 1, 1], caps)
    full = obj.to_tensor()
    got = obj.to_tensor_coarse(1)
    assert np.abs(got - block_mean(full, (5, 2, 5))).max() <= 1e-12 * np.abs(full).max()


def _idct_mean_ref(x, block):
    from scipy.fft import idct
    rec = idct(x.astype(np.float64), type=2, axis=-1, norm="ortho")
    return rec.reshape(*x.shape[:-1], x.shape[-1] // block, block).mean(axis=-1)


@pytest.mark.parametrize("n", [20, 50, 64, 1920])
def test_idct_block_mean_last_axis_against_scipy(n):
    from imgcompressionmps import _ops
    rng = np.random.default_rng(n)
    blocks = [b for b in range(1, n + 1) if n % b == 0]
    cases = [(np.float64, 37), (np.float32, 37), (np.float32, -(-(1 << 20) // n))]   # below / at the tcgen05 threshold
    for dtype, lines in cases:
        x = rng.standard_normal((lines, n)).astype(dtype)
        dev = torch.from_numpy(x).cuda()
        for b in blocks:
            got = _ops.idct_block_mean_last_axis(dev, b).cpu().numpy()
            ref = _idct_mean_ref(x, b)
            assert got.shape == ref.shape and got.dtype == x.dtype
            tol = (1e-12 if dtype == np.float64 else 1e-5) * float(np.abs(_idct_mean_ref(x, 1)).max())
            assert np.abs(got - ref).max() <= tol, (dtype, lines, b, float(np.abs(got - ref).max()), tol)
        full = _ops.dct_last_axis(dev, inverse=True)
        one = _ops.idct_block_mean_last_axis(dev, 1)
        assert float((one - full).abs().max()) <= (1e-12 if dtype == np.float64 else 1e-6) * float(full.abs().max())


def test_idct_block_mean_rejects_a_block_that_does_not_divide():
    from imgcompressionmps import _ops
    x = torch.zeros((4, 50), dtype=torch.float64, device="cuda")
    for b in (0, 3, 7, 51, -5):
        with pytest.raises(ValueError):
            _ops.idct_block_mean_last_axis(x, b)


def test_coarse_memory_is_bounded_by_the_result(NDMPS):
    """256^3 float32 at chi = 128 averaged over 2 levels (a 64^3 result), in a fresh thread with its own context: the
    arena's high-water mark and torch's peak allocation during the call both stay below 1/8 of the 64 MB tensor; the
    full reconstruction followed by a mean would need the whole tensor twice."""
    from imgcompressionmps import _native as N
    shape = (256, 256, 256)
    obj = NDMPS.from_tensor(smooth(shape, seed=5).astype(np.float32), max_bond=128)
    full = obj.to_tensor_device().double()
    want = full.view(64, 4, 64, 4, 64, 4).mean(dim=(1, 3, 5)).cpu().numpy()
    scale = float(full.abs().max())
    del full
    torch.cuda.synchronize()
    result = {}

    def run():
        try:
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            out = obj.to_tensor_coarse_device(2)
            torch.cuda.synchronize()
            result["peak"] = torch.cuda.max_memory_allocated() - base
            obj.to_tensor_coarse_device(2, (0, 0, 0))        # the high-water mark folds in at the next reset
            torch.cuda.synchronize()
            result["out"] = out.cpu().numpy()
            result["ws"] = N.context().stat("workspace_bytes")
        except Exception as exc:                            # surfaced in the main thread
            result["error"] = exc

    t = threading.Thread(target=run)
    t.start()
    t.join()
    if "error" in result:
        raise result["error"]
    tensor_bytes = 4 * 256 ** 3
    assert result["out"].shape == (64, 64, 64)
    assert 0 < result["ws"] < tensor_bytes / 8, result["ws"]
    assert 0 < result["peak"] < tensor_bytes / 8, result["peak"]
    assert np.abs(result["out"] - want).max() <= 1e-5 * scale
