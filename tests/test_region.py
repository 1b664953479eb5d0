"""Host-side index math of the region decode (no device work): the flat site-order index the region path reads
for every voxel of a box equals the one the reference's encoding map gives, and the index helper of
``NDMPS.to_tensor_region`` selects the boxes numpy's basic indexing selects."""
import numpy as np
import pytest

from imgcompressionmps import _native as N
from imgcompressionmps import _ops
from imgcompressionmps.utils.core import gen_encoding_map, get_factorlist

SHAPES = [(8, 9), (4, 6), (12, 18, 10), (16, 16, 8, 20), (30, 40, 50), (7,), (1, 4), (64, 64), (64, 64, 64)]


def _site_flat(shape):
    dims, enc = gen_encoding_map(shape)
    flat = np.zeros(shape, dtype=np.int64)
    for lvl in range(len(dims)):
        flat = flat * int(dims[lvl]) + enc[lvl]
    return flat


def _boxes(shape):
    """full; an int on each axis; one voxel; an unaligned sub-box; a box whose low parts wrap across a block
    boundary; an empty range"""
    nd = len(shape)
    full = tuple(slice(None) for _ in shape)
    out = [("full", full)]
    for a, n in enumerate(shape):
        out.append((f"int{a}", full[:a] + (n // 2,) + full[a + 1:]))
    out.append(("voxel", tuple(n - 1 - n // 3 for n in shape)))
    out.append(("unaligned", tuple(slice(n // 5, max(n // 5 + 1, n - n // 4)) for n in shape)))
    # a narrow range that starts just below the middle of the axis: inside the low part it runs past the
    # block boundary at n / 2 (for even extents), so the set of low parts wraps
    out.append(("wrap", tuple(slice(max(n // 2 - 1, 0), min(n // 2 + 2, n)) for n in shape)))
    out.append(("empty", full[:nd - 1] + (slice(3, 3),)))
    return out


def _lo_hi(shape, index):
    lo, hi, _ = _ops.region_box(shape, index)
    return lo, hi


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_region_offsets_match_encoding_map(shape):
    factors, _ = get_factorlist(shape)
    plan = N.Plan(shape, factors)
    flat = _site_flat(shape)
    L = len(plan.site_dims)
    total = int(np.prod(shape))
    for name, index in _boxes(shape):
        lo, hi = _lo_hi(shape, index)
        info, offs = plan.region_debug(lo, hi)
        box = tuple(slice(l, h) for l, h in zip(lo, hi))
        want = flat[box].reshape(-1)
        assert info["s"] == 1 if L == 1 else 1 <= info["s"] <= L - 1, (name, info)
        if want.size == 0:
            assert info["rows"] == 0 and info["cols"] == 0 and offs.size == 0, name
            continue
        assert np.array_equal(offs, want), name
        # |H| |C| <= 3^ndim |box|, and the split's rows / columns never exceed the full ones
        rows_full = int(np.prod(plan.site_dims[:info["s"]]))
        assert info["rows"] * info["cols"] <= 3 ** len(shape) * want.size, name
        assert info["rows"] <= rows_full and info["cols"] <= total // rows_full, name
        if name == "full":
            assert info["rows"] * info["cols"] == total


@pytest.mark.parametrize("shape", [(64, 64, 64), (30, 40, 50), (16, 16, 8, 20)], ids=lambda s: "x".join(map(str, s)))
def test_slices_and_aligned_boxes_keep_exactly_the_box(shape):
    """For a slice, and for ranges that cover whole blocks of the split, H x C is the box itself."""
    factors, _ = get_factorlist(shape)
    plan = N.Plan(shape, factors)
    for a, n in enumerate(shape):
        index = tuple(slice(None) for _ in shape[:a]) + (n // 3,)
        lo, hi = _lo_hi(shape, index)
        info, offs = plan.region_debug(lo, hi)
        assert info["rows"] * info["cols"] == offs.size, (a, info)


def test_region_offsets_random_boxes():
    rng = np.random.default_rng(7)
    for shape in [(12, 18, 10), (30, 40, 50), (64, 64, 64), (16, 16, 8, 20), (24, 36)]:
        factors, _ = get_factorlist(shape)
        plan = N.Plan(shape, factors)
        flat = _site_flat(shape)
        for _ in range(20):
            lo = [int(rng.integers(0, n)) for n in shape]
            hi = [int(rng.integers(l + 1, n + 1)) for l, n in zip(lo, shape)]
            info, offs = plan.region_debug(lo, hi)
            assert np.array_equal(offs, flat[tuple(slice(l, h) for l, h in zip(lo, hi))].reshape(-1)), (shape, lo, hi)
            assert info["rows"] * info["cols"] <= 3 ** len(shape) * offs.size


def test_region_debug_rejects_a_box_outside_the_volume():
    shape = (8, 9)
    factors, _ = get_factorlist(shape)
    plan = N.Plan(shape, factors)
    for lo, hi in [([0, 0], [9, 9]), ([-1, 0], [2, 2]), ([3, 0], [2, 9])]:
        with pytest.raises(ValueError):
            plan.region_debug(lo, hi)


_INDEX_CASES = [
    (5, 7, 9),
    (slice(None),),
    (slice(2, 5),),
    (slice(-3, None), 1),
    (Ellipsis, 2),
    (1, Ellipsis),
    (1, Ellipsis, -1),
    (slice(4, 100), slice(-100, 2), slice(6, 2)),
    (np.int64(3), slice(None, None, 1)),
    (0, 0, 0),
    (-6, -9, -11),
    (Ellipsis,),
    (),
    (slice(None), slice(3, 3)),
]


@pytest.mark.parametrize("index", _INDEX_CASES + [3, slice(1, 4), Ellipsis], ids=repr)
def test_index_helper_matches_numpy_shapes(index):
    shape = (6, 9, 11)
    want = np.empty(shape)[index].shape
    lo, hi, got = _ops.region_box(shape, index)
    assert got == want
    ramp = np.arange(int(np.prod(shape))).reshape(shape)
    box = ramp[tuple(slice(l, h) for l, h in zip(lo, hi))]
    assert np.array_equal(box.reshape(want), ramp[index])


@pytest.mark.parametrize("index", [(6,), (0, 9), (0, 0, -12), (1, 2, 3, 4), (Ellipsis, Ellipsis), (1.0,), ("a",),
                                   (slice(1.5, 3),)], ids=repr)
def test_index_helper_raises_numpys_error_types(index):
    shape = (6, 9, 11)
    with pytest.raises(Exception) as np_err:
        np.empty(shape)[index]
    with pytest.raises(type(np_err.value)):
        _ops.region_box(shape, index)


@pytest.mark.parametrize("index", [(slice(None, None, 2),), (slice(None, None, -1),), (slice(0, 4, 0),), (None,),
                                   (np.array([1, 2]),), (True,)], ids=repr)
def test_index_helper_rejects_what_a_box_cannot_express(index):
    with pytest.raises(ValueError):
        _ops.region_box((6, 9, 11), index)
