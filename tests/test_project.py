"""Host-side index math of the intensity projection (no device work): for every output element and every position
along the projected axis, the block plan of ``ndmps_project_region`` reads the site-order index the reference's
encoding map gives for that voxel, and exactly one block reads it, whatever the block bound; and the argument rules of
``NDMPS.project``, which are checked before anything touches the device."""
import numpy as np
import pytest

from imgcompressionmps import _native as N
from imgcompressionmps import _ops
from imgcompressionmps.utils.core import get_factorlist
from test_region import SHAPES, _boxes, _site_flat


def _plan(shape):
    factors, _ = get_factorlist(shape)
    return N.Plan(shape, factors)


def _block_bounds(plan, lo, hi):
    """block bounds in elements of T: one axis-0 high part, three, and all of T in one block"""
    info, _, _ = plan.project_debug(lo, hi, 0, 1)
    per_h = info["rows"] * info["cols"] // info["blocks"]        # a bound of 1 gives one high part per block
    return {"one": 1, "three": 3 * per_h, "all": info["rows"] * info["cols"]}


def check_projection_offsets(shape, lo, hi):
    plan = _plan(shape)
    flat = _site_flat(shape)
    box = flat[tuple(slice(l, h) for l, h in zip(lo, hi))]
    for name, bound in _block_bounds(plan, lo, hi).items():
        for axis in range(len(shape)):
            info, offs, blocks = plan.project_debug(lo, hi, axis, bound)
            want = np.moveaxis(box, axis, -1).reshape(-1, box.shape[axis])
            assert np.array_equal(offs, want), (shape, lo, hi, axis, name)
            assert (blocks >= 0).all(), (shape, lo, hi, axis, name)        # -1: no block, -2: more than one
            # blocks are ranges of axis-0 positions, in order
            per_i0 = np.moveaxis(blocks.reshape([hi[a] - lo[a] for a in range(len(shape)) if a != axis]
                                                + [hi[axis] - lo[axis]]), -1, axis)
            b0 = per_i0.reshape(hi[0] - lo[0], -1)
            assert (b0 == b0[:, :1]).all() and (np.diff(b0[:, 0]) >= 0).all(), (shape, lo, hi, axis, name)
            assert int(b0.max()) + 1 == info["blocks"], (shape, lo, hi, axis, name)
            if name == "all" or len(plan.site_dims) == 1:
                assert info["blocks"] == 1
            if name == "one" and len(plan.site_dims) > 1:
                # one axis-0 high part per block, and so as many blocks as the split's high parts the box touches
                g0 = int(np.prod(np.array(plan.factors)[info["s"]:, 0]))
                assert info["blocks"] == (hi[0] - 1) // g0 - lo[0] // g0 + 1


@pytest.mark.parametrize("shape", SHAPES + [(5, 1, 3)], ids=lambda s: "x".join(map(str, s)))
def test_projection_offsets_match_encoding_map(shape):
    for name, index in _boxes(shape):
        lo, hi, _ = _ops.region_box(shape, index)
        if any(h == l for l, h in zip(lo, hi)):
            continue
        check_projection_offsets(shape, lo, hi)


@pytest.mark.parametrize("shape", [(4096,), (3000,), (1 << 16,)], ids=lambda s: "x".join(map(str, s)))
def test_projection_offsets_of_multi_level_1d_signals(shape):
    """A 1-D signal of several levels splits into blocks along its only axis, which is also the projected one: each
    block reads its own positions and no other."""
    plan = _plan(shape)
    assert len(plan.site_dims) > 1
    assert plan.project_debug([0], list(shape), 0, 1)[0]["blocks"] > 1
    for name, index in _boxes(shape):
        lo, hi, _ = _ops.region_box(shape, index)
        if any(h == l for l, h in zip(lo, hi)):
            continue
        check_projection_offsets(shape, lo, hi)


def test_projection_offsets_random_boxes():
    rng = np.random.default_rng(3)
    for shape in [(12, 18, 10), (30, 40, 50), (16, 16, 8, 20), (24, 36)]:
        for _ in range(6):
            lo = [int(rng.integers(0, n)) for n in shape]
            hi = [int(rng.integers(l + 1, n + 1)) for l, n in zip(lo, shape)]
            check_projection_offsets(shape, lo, hi)


def test_projection_debug_rejects_what_the_device_path_rejects():
    plan = _plan((8, 9))
    for lo, hi, axis in [([0, 0], [9, 9], 0), ([0, 0], [8, 9], 2), ([0, 0], [8, 9], -1), ([3, 0], [3, 9], 0)]:
        with pytest.raises(ValueError):
            plan.project_debug(lo, hi, axis, 1 << 20)
    info, offs, blocks = plan.project_debug([3, 0], [3, 9], 1, 1 << 20)    # empty on another axis: nothing to read
    assert info["blocks"] == 0 and offs.size == 0 and blocks.size == 0


# ---- argument rules of NDMPS.project (checked before the device is touched) ------------------------------------------
class _Stub:
    """An NDMPS with a shape and a mode but no cores: the argument checks run, nothing else can."""

    def __new__(cls, shape, mode="other"):
        from imgcompressionmps.core.ndmps import NDMPS
        obj = NDMPS(mode=mode)
        obj._shape = tuple(shape)
        return obj


def test_argument_rules_need_no_device():
    obj = _Stub((6, 9, 11))
    for op in ("mean", "sum", "argmax", None, "MAX"):
        with pytest.raises(ValueError):
            obj.project(0, op)
    for axis in (3, -4):
        with pytest.raises(ValueError):
            obj.project(axis)
    with pytest.raises(ValueError):                                       # the ints drop axes 0 and 2: one axis left
        obj.project(1, index=(2, slice(None), 4))
    with pytest.raises(ValueError):                                       # 0-d indexed result
        obj.project(0, index=(1, 2, 3))
    with pytest.raises(ValueError):                                       # empty along the projected axis
        obj.project(1, index=(slice(None), slice(4, 4)))
    with pytest.raises(ValueError):
        obj.project(-1, index=(Ellipsis, slice(4, 2), 0))
    for axis in (1.0, "0", True):
        with pytest.raises(TypeError):
            obj.project(axis)
    with pytest.raises(IndexError):
        obj.project(0, index=(6,))
    with pytest.raises(ValueError):
        obj.project(0, index=(slice(None, None, 2),))
    # valid arguments: an unknown mode returns None after the checks
    assert obj.project(0) is None and obj.project_device(-1, "min", (1,)) is None
    assert obj.project(0, index=(slice(None), slice(3, 3))) is None       # empty on another axis


@pytest.mark.parametrize("index,axis", [((), 0), ((), -1), ((2,), 0), ((2,), 1), ((slice(1, 4), 5), 0),
                                        ((Ellipsis, 3), -2), ((slice(1, 4), 5, slice(2, 9)), -1), ((0, 0), 0),
                                        ((slice(None), slice(3, 3)), 0)], ids=repr)
def test_axis_maps_to_the_volume_axis_numpy_reduces(index, axis):
    shape = (6, 9, 11)
    obj = _Stub(shape)
    lo, hi, vaxis, res_shape = obj._projection_args(axis, "max", index)
    ramp = np.arange(int(np.prod(shape))).reshape(shape)
    want = np.max(ramp[index], axis=axis)
    assert res_shape == want.shape
    box = ramp[tuple(slice(l, h) for l, h in zip(lo, hi))]
    assert np.array_equal(np.max(box, axis=vaxis).reshape(res_shape), want)


def test_region_box_axes_names_the_kept_axes():
    assert _ops.region_box_axes((6, 9, 11), (2,))[3] == (1, 2)
    assert _ops.region_box_axes((6, 9, 11), (Ellipsis, 3))[3] == (0, 1)
    assert _ops.region_box_axes((6, 9, 11), (slice(1, 2), -1))[3] == (0, 2)
    assert _ops.region_box_axes((6, 9, 11), (1, 2, 3))[3] == ()
    assert _ops.region_box_axes((6, 9, 11), (1, 2))[:3] == _ops.region_box((6, 9, 11), (1, 2))
