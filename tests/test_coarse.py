"""Host-side layout of the block-mean (coarse) decode, no device work: the coarse shape and factor table the library
decides, its decode offsets, a float64 numpy restatement of the marginalisation that must give the block mean of the
dense reconstruction when decoded with that table, and the argument rules of ``NDMPS.to_tensor_coarse``."""
import numpy as np
import pytest

from imgcompressionmps import _ops
from imgcompressionmps.core.ndmps import NDMPS
from imgcompressionmps.utils.core import get_factorlist

SHAPES = [(8, 9), (4, 6), (7,), (1, 4), (12, 18, 10), (16, 16, 8, 20), (30, 40, 50), (64, 64, 64), (1920, 1080, 64)]


def level_cases(shape):
    """0, 1, L on every axis, and a per-axis mix with L on the first axis"""
    L = get_factorlist(shape)[0].shape[0]
    mix = tuple(L if a == 0 else a % (L + 1) for a in range(len(shape)))
    return [0, min(1, L), L, mix]


def derive(shape, levels):
    """(coarse shape, coarse factor table, block) from get_factorlist, as the block mean defines them"""
    f, _ = get_factorlist(shape)
    L, n = f.shape
    k = [int(levels)] * n if np.isscalar(levels) else [int(v) for v in levels]
    block = tuple(int(np.prod(f[L - k[a]:, a])) for a in range(n))
    cf = f.copy()
    for a in range(n):
        cf[L - k[a]:, a] = 1
    cf = cf[:max(1, L - min(k))]
    return tuple(s // b for s, b in zip(shape, block)), cf, block


def site_flat(shape, factors):
    """flat site-order index of every voxel for an explicit factor table (gen_encoding_map with given factors)"""
    L, n = factors.shape
    flat = np.zeros(shape, dtype=np.int64)
    dims = np.prod(factors, axis=1)
    digits = []
    for a in range(n):
        coord = np.arange(shape[a], dtype=np.int64)
        below, per = 1, [None] * L
        for lvl in range(L - 1, -1, -1):
            per[lvl] = (coord // below) % int(factors[lvl, a])
            below *= int(factors[lvl, a])
        digits.append(per)
    for lvl in range(L):
        site = np.zeros(shape, dtype=np.int64)
        for a in range(n):
            view = [1] * n
            view[a] = shape[a]
            site = site * int(factors[lvl, a]) + digits[a][lvl].reshape(view)
        flat = flat * int(dims[lvl]) + site
    return flat


def block_mean(x, block):
    split = []
    for s, b in zip(x.shape, block):
        split += [s // b, b]
    return x.reshape(split).mean(axis=tuple(range(1, 2 * x.ndim, 2)))


def _ids(s):
    return "x".join(map(str, s))


@pytest.mark.parametrize("shape", SHAPES, ids=_ids)
def test_coarse_plan_matches_factorlist_derivation(shape):
    obj = NDMPS()
    obj._shape = shape
    for levels in level_cases(shape):
        cshape, cf, _ = derive(shape, levels)
        plan = _ops.coarse_plan(shape, levels)
        assert plan.shape == cshape and obj.coarse_shape(levels) == cshape, levels
        assert np.array_equal(plan.factors, cf), (levels, plan.factors, cf)
        assert plan.levels == cf.shape[0] and plan.site_dims == [int(d) for d in np.prod(cf, axis=1)]


def test_coarse_shapes_of_the_documented_examples():
    assert _ops.coarse_plan((512, 512, 512), 3).shape == (64, 64, 64)
    assert _ops.coarse_plan((30, 40, 50), 1).shape == (6, 20, 10)
    assert _ops.coarse_plan((1920, 1080, 64), (1, 1, 0)).shape == (384, 540, 64)
    assert _ops.coarse_plan((1920, 1080, 64), (2, 2, 0)).shape == (96, 180, 64)
    L = get_factorlist((30, 40, 50))[0].shape[0]
    plan = _ops.coarse_plan((30, 40, 50), L)
    assert plan.shape == (1, 1, 1) and plan.levels == 1 and plan.site_dims == [1]


@pytest.mark.parametrize("shape", [s for s in SHAPES if np.prod(s) <= 1 << 18], ids=_ids)
def test_coarse_plan_decode_offsets(shape):
    for levels in level_cases(shape):
        cshape, cf, _ = derive(shape, levels)
        plan = _ops.coarse_plan(shape, levels)
        total = int(np.prod(cshape))
        assert np.array_equal(plan.debug_offsets(True, 0, total), site_flat(cshape, cf).reshape(-1)), levels


def random_mps(dims, rng):
    L = len(dims)
    if L == 1:
        return [rng.standard_normal(dims[0])], []
    ranks = [int(rng.integers(1, 6)) for _ in range(L - 1)]
    cores = [rng.standard_normal((dims[0], ranks[0]))]
    cores += [rng.standard_normal((ranks[i - 1], dims[i], ranks[i])) for i in range(1, L - 1)]
    cores.append(rng.standard_normal((ranks[-1], dims[-1])))
    return cores, ranks


def contract(cores):
    out = np.asarray(cores[0]).reshape(1, -1, cores[0].shape[-1] if len(cores) > 1 else 1)
    acc = out.reshape(-1, out.shape[-1])
    for c in cores[1:]:
        c3 = c if c.ndim == 3 else c.reshape(c.shape[0], c.shape[1], 1)
        acc = (acc @ c3.reshape(c3.shape[0], -1)).reshape(-1, c3.shape[2])
    return acc.reshape(-1)


def marginalize_np(cores, factors, levels):
    """float64 restatement: site l averaged over its averaged digits, the fully averaged suffix folded into v"""
    L, n = factors.shape
    k = [int(levels)] * n if np.isscalar(levels) else list(levels)
    full3 = []
    for l, c in enumerate(cores):
        rl = 1 if l == 0 else c.shape[0]
        rr = 1 if l == L - 1 else c.shape[-1]
        c = c.reshape(rl, *[int(f) for f in factors[l]], rr)
        avg = tuple(1 + a for a in range(n) if l >= L - k[a])
        full3.append(c.mean(axis=avg).reshape(rl, -1, rr) if avg else c.reshape(rl, -1, rr))
    Lk = max(1, L - min(k))
    v = np.ones(1)
    for l in range(L - 1, Lk - 1, -1):
        v = full3[l][:, 0, :] @ v
    out = full3[:Lk]
    out[-1] = out[-1] @ v if Lk < L else out[-1][..., 0]
    out[0] = out[0][0]
    return out


@pytest.mark.parametrize("shape", [(8, 9), (4, 6), (7,), (1, 4), (12, 18, 10), (16, 16, 8, 20), (30, 40, 50)], ids=_ids)
def test_numpy_marginalization_decoded_with_the_coarse_plan_is_the_block_mean(shape):
    rng = np.random.default_rng(sum(shape))
    factors, _ = get_factorlist(shape)
    dims = [int(d) for d in np.prod(factors, axis=1)]
    flat = site_flat(shape, factors)
    for trial in range(3):
        cores, _ = random_mps(dims, rng)
        full = contract(cores)[flat]
        for levels in level_cases(shape):
            plan = _ops.coarse_plan(shape, levels)
            _, _, block = derive(shape, levels)
            red = marginalize_np(cores, factors, levels)
            assert len(red) == plan.levels
            coarse = contract(red)
            assert coarse.size == int(np.prod(plan.site_dims))
            vol = coarse[plan.debug_offsets(True, 0, plan.total)].reshape(plan.shape)
            want = block_mean(full, block)
            assert np.abs(vol - want).max() <= 1e-12 * max(1.0, np.abs(full).max()), (trial, levels)


def test_levels_argument_rules():
    shape = (30, 40, 50)
    L = get_factorlist(shape)[0].shape[0]
    assert _ops.coarse_levels(shape, np.int64(1)) == (1, 1, 1)
    assert _ops.coarse_levels(shape, np.array([1, 0, L])) == (1, 0, L)
    assert _ops.coarse_levels(shape, [np.int32(0), 1, 2]) == (0, 1, 2)
    for bad in (True, np.bool_(True), 1.0, "1", None, [1, 1.0, 0], [True, 0, 0], np.float64(1)):
        with pytest.raises(TypeError):
            _ops.coarse_levels(shape, bad)
    for bad in (-1, L + 1, [1, 1], [0, 0, 0, 0], [0, -1, 0], [0, 0, L + 1]):
        with pytest.raises(ValueError):
            _ops.coarse_levels(shape, bad)
    plan = _ops.plan_for(shape)
    for bad in ([-1, 0, 0], [0, 0, L + 1]):
        with pytest.raises(ValueError):
            plan.coarse(bad)


def _unknown_mode(shape):
    obj = NDMPS(mode="other")
    obj._shape = shape
    return obj


def test_public_methods_check_levels_and_index_before_the_mode():
    """Argument errors come before anything touches the device; a mode other than Std / DCT then returns None."""
    obj = _unknown_mode((30, 40, 50))
    assert obj.coarse_shape(1) == (6, 20, 10)
    with pytest.raises(TypeError):
        obj.to_tensor_coarse(1.5)
    with pytest.raises(ValueError):
        obj.to_tensor_coarse_device([1, 1])
    # the index applies to the coarse shape (6, 20, 10)
    for bad in ((6,), (0, 20), (0, 0, -11), (0, 0, 0, 0)):
        with pytest.raises(IndexError):
            obj.to_tensor_coarse(1, bad)
    with pytest.raises(ValueError):
        obj.to_tensor_coarse(1, (slice(None, None, 2),))
    for ok in (None, (5,), (slice(2, 4), -20), (Ellipsis, 9), ()):
        assert obj.to_tensor_coarse(1, ok) is None and obj.to_tensor_coarse_device(1, ok) is None


@pytest.mark.parametrize("index", [None, (1,), (slice(1, 4), Ellipsis, -1), (0, 0, slice(3, 3))], ids=repr)
def test_coarse_index_box_matches_numpy_on_the_coarse_shape(index):
    cshape = _ops.coarse_plan((30, 40, 50), 1).shape
    lo, hi, got = _ops.region_box(cshape, () if index is None else index)
    ramp = np.arange(int(np.prod(cshape))).reshape(cshape)
    want = ramp if index is None else ramp[index]
    assert got == want.shape
    assert np.array_equal(ramp[tuple(slice(l, h) for l, h in zip(lo, hi))].reshape(got), want)
