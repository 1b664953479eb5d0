"""Thin torch-tensor wrappers over the C ABI (``include/ndmps.h``).

Every function here launches this repo's own CUDA kernels on torch's current
stream; torch only provides the device buffers.  Nothing falls back to torch math.
"""
from __future__ import annotations

import ctypes as C
from functools import lru_cache

import numpy as np

from . import _native as N
from .utils.core import get_factorlist


def _torch():
    import torch
    return torch


def _dev(t, what="tensor"):
    if not t.is_cuda:
        raise ValueError(f"{what} must live on the CUDA device")
    if not t.is_contiguous():
        raise ValueError(f"{what} must be contiguous")
    return t


@lru_cache(maxsize=64)
def plan_for(shape) -> N.Plan:
    shape = tuple(int(s) for s in shape)
    factors, _ = get_factorlist(shape)
    return N.Plan(shape, factors)


def coarse_levels(shape, levels) -> tuple:
    """Validated per-axis digit counts of a block mean: ``levels`` is an int (every axis) or a sequence of ``ndim``
    ints, each in ``0 ..= L`` (L = the levels of ``get_factorlist(shape)``); numpy integers are accepted.  A bool or a
    non-integer raises ``TypeError``, a wrong length or a value out of range ``ValueError``."""
    import operator
    shape = tuple(int(s) for s in shape)
    L = int(get_factorlist(shape)[0].shape[0])

    def one(v):
        if isinstance(v, (bool, np.bool_)) or not hasattr(v, "__index__"):
            raise TypeError(f"levels: {v!r} is not an integer")
        return operator.index(v)

    if isinstance(levels, (list, tuple, np.ndarray)):
        ks = tuple(one(v) for v in levels)
        if len(ks) != len(shape):
            raise ValueError(f"levels: {len(ks)} values for a {len(shape)}-dimensional volume")
    else:
        ks = (one(levels),) * len(shape)
    if any(not 0 <= k <= L for k in ks):
        raise ValueError(f"levels: {ks} outside 0..{L} (the volume has {L} levels)")
    return ks


@lru_cache(maxsize=64)
def _coarse_plan(shape, ks) -> N.Plan:
    return plan_for(shape).coarse(ks)


def coarse_plan(shape, levels) -> N.Plan:
    """Plan of the block mean of a volume of ``shape`` over the finest ``levels`` digits of each axis
    (``ndmps_plan_coarse``; its ``shape`` is the coarse shape)."""
    shape = tuple(int(s) for s in shape)
    return _coarse_plan(shape, coarse_levels(shape, levels))


# ---- K1 ---------------------------------------------------------------------------
def encode(volume, scale: float = 1.0, plan=None):
    """volume (original shape, device) -> dense array shaped by the site dims."""
    torch = _torch()
    plan = plan or plan_for(tuple(volume.shape))
    _dev(volume, "volume")
    out = torch.empty(plan.site_dims, dtype=volume.dtype, device=volume.device)
    N.check(N.load_library().ndmps_encode(N.handle(), plan.handle, N.ptr(volume), N.ptr(out),
                                          N.dtype_code(volume.dtype), float(scale)), "ndmps_encode")
    return out


def decode(dense, shape, plan=None):
    torch = _torch()
    plan = plan or plan_for(tuple(shape))
    _dev(dense, "dense")
    if dense.numel() != plan.total:
        raise ValueError("dense array does not match the volume shape")
    out = torch.empty(plan.shape, dtype=dense.dtype, device=dense.device)
    N.check(N.load_library().ndmps_decode(N.handle(), plan.handle, N.ptr(dense), N.ptr(out),
                                          N.dtype_code(dense.dtype)), "ndmps_decode")
    return out


# ---- reductions ---------------------------------------------------------------------
def sumsq(x) -> float:
    _dev(x)
    out = C.c_double()
    N.check(N.load_library().ndmps_sumsq(N.handle(), N.ptr(x), x.numel(), N.dtype_code(x.dtype), C.byref(out)),
            "ndmps_sumsq")
    return out.value


def minmax(tensors) -> np.ndarray:
    tensors = [_dev(t) for t in tensors]
    if not tensors:
        return np.zeros((0, 2))
    code = N.dtype_code(tensors[0].dtype)
    out = np.empty((len(tensors), 2), dtype=np.float64)
    N.check(N.load_library().ndmps_minmax(N.handle(), N.ptr_array(tensors), N.i64_array([t.numel() for t in tensors]),
                                          len(tensors), code, out.ctypes.data_as(N.p_f64)), "ndmps_minmax")
    return out


def psnr_terms(a, b):
    _dev(a), _dev(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        raise ValueError("PSNR operands must share shape and dtype")
    out = (C.c_double * 2)()
    N.check(N.load_library().ndmps_psnr_terms(N.handle(), N.ptr(a), N.ptr(b), a.numel(), N.dtype_code(a.dtype), out),
            "ndmps_psnr_terms")
    return out[0], out[1]


# ---- K11 ---------------------------------------------------------------------------
def dct_last_axis(x, inverse: bool = False):
    torch = _torch()
    _dev(x)
    n = int(x.shape[-1])
    out = torch.empty_like(x)
    N.check(N.load_library().ndmps_dct_last_axis(N.handle(), N.ptr(x), N.ptr(out), x.numel() // n, n,
                                                 int(bool(inverse)), N.dtype_code(x.dtype)), "ndmps_dct_last_axis")
    return out


def idct_block_mean_last_axis(x, block: int):
    """Block mean (``block`` elements) of the orthonormal inverse DCT along the last axis, without the full lines."""
    torch = _torch()
    _dev(x)
    n = int(x.shape[-1])
    block = int(block)
    out = torch.empty(tuple(x.shape[:-1]) + (n // block if block >= 1 else 0,), dtype=x.dtype, device=x.device)
    N.check(N.load_library().ndmps_idct_block_mean_last_axis(N.handle(), N.ptr(x), N.ptr(out), x.numel() // n, n, block,
                                                             N.dtype_code(x.dtype)), "ndmps_idct_block_mean_last_axis")
    return out


# ---- building blocks ---------------------------------------------------------------
def gram(m, side: int = 0):
    torch = _torch()
    _dev(m)
    rows, cols = int(m.shape[0]), int(m.shape[1])
    n = rows if side == 0 else cols
    g = torch.empty((n, n), dtype=torch.float64, device=m.device)
    N.check(N.load_library().ndmps_gram(N.handle(), N.ptr(m), rows, cols, cols, N.dtype_code(m.dtype), int(side),
                                        N.ptr(g)), "ndmps_gram")
    return g


def eigh(a):
    """Eigen-decomposition of a symmetric float64 matrix (descending); returns (evals, evecs, sweeps)."""
    torch = _torch()
    _dev(a)
    if a.dtype != torch.float64 or a.ndim != 2 or a.shape[0] != a.shape[1]:
        raise ValueError("eigh expects a square float64 matrix")
    n = int(a.shape[0])
    work = a.clone()
    evals = torch.empty(n, dtype=torch.float64, device=a.device)
    evecs = torch.empty((n, n), dtype=torch.float64, device=a.device)
    sweeps = C.c_int(0)
    N.check(N.load_library().ndmps_eigh(N.handle(), N.ptr(work), n, N.ptr(evals), N.ptr(evecs), C.byref(sweeps)),
            "ndmps_eigh")
    return evals, evecs, sweeps.value


def eigh_topk(a, k: int):
    """Leading k eigenpairs of a symmetric PSD float64 matrix; returns (evals[k] descending, evecs[n, k], trace, health)."""
    torch = _torch()
    _dev(a)
    if a.dtype != torch.float64 or a.ndim != 2 or a.shape[0] != a.shape[1]:
        raise ValueError("eigh_topk expects a square float64 matrix")
    n, k = int(a.shape[0]), int(k)
    a = a.contiguous()
    out = torch.empty(k + 2, dtype=torch.float64, device=a.device)
    evecs = torch.empty((n, k), dtype=torch.float64, device=a.device)
    N.check(N.load_library().ndmps_eigh_topk(N.handle(), N.ptr(a), n, k, N.ptr(out), N.ptr(evecs)), "ndmps_eigh_topk")
    host = out.cpu()
    return out[:k], evecs, float(host[k]), int(host[k + 1])


def gemm(a, b, out_dtype=None, alpha: float = 1.0):
    """a @ b for 2-D (possibly transposed-view) device tensors through ndmps_gemm."""
    torch = _torch()
    m, k = a.shape
    k2, n = b.shape
    if k != k2:
        raise ValueError("gemm: inner dimensions differ")
    out_dtype = out_dtype or a.dtype
    c = torch.empty((m, n), dtype=out_dtype, device=a.device)
    N.check(N.load_library().ndmps_gemm(N.handle(), m, n, k, float(alpha),
                                        N.ptr(a), N.dtype_code(a.dtype), a.stride(0), a.stride(1),
                                        N.ptr(b), N.dtype_code(b.dtype), b.stride(0), b.stride(1),
                                        N.ptr(c), N.dtype_code(out_dtype), n), "ndmps_gemm")
    return c


# ---- sweep / truncation / contraction -------------------------------------------------
def bond_bounds(dims, max_bond=None):
    """Upper bound of every bond: min(prod left, prod right, max_bond)."""
    L = len(dims)
    out = []
    left = 1
    for i in range(L - 1):
        left *= int(dims[i])
        right = 1
        for d in dims[i + 1:]:
            right *= int(d)
        bound = min(left, right)
        # a bond can also never exceed (previous bond * d_i)
        if out:
            bound = min(bound, out[-1] * int(dims[i]))
        if max_bond:
            bound = min(bound, int(max_bond))
        out.append(bound)
    return out


def core_shape(i, L, dims, ranks):
    if L == 1:
        return (int(dims[0]),)
    if i == 0:
        return (int(dims[0]), int(ranks[0]))
    if i == L - 1:
        return (int(ranks[L - 2]), int(dims[L - 1]))
    return (int(ranks[i - 1]), int(dims[i]), int(ranks[i]))


def _trim_mode(cutoff_mode, renorm):
    """Mode code and renorm power of a sweep; ``renorm=None`` takes the mode's default."""
    mode = N.CUTOFF_MODES[cutoff_mode]
    default = {N.CUT_RSUM2: 2, N.CUT_SUM2: 2, N.CUT_RSUM1: 1, N.CUT_SUM1: 1}.get(mode, 0)
    return mode, int(default if renorm is None else renorm)


def _sweep_args(dims, cutoff, cutoff_mode, renorm, max_bond, like):
    """Arguments cutoff .. svals_stride of both sweep entry points, and the buffers (like ``like``) they point to."""
    torch = _torch()
    L = len(dims)
    bounds = bond_bounds(dims, max_bond)
    caps = [int(np.prod(core_shape(i, L, dims, bounds), dtype=np.int64)) for i in range(L)]
    bufs = [torch.empty(c, dtype=like.dtype, device=like.device) for c in caps]
    ranks = (C.c_int64 * max(L - 1, 1))()
    svals = np.zeros((max(L - 1, 1), max(bounds) if bounds else 1), dtype=np.float64)
    mode, renorm = _trim_mode(cutoff_mode, renorm)
    args = (float(cutoff), mode, int(max_bond or 0), renorm, N.ptr_array(bufs), N.i64_array(caps), ranks,
            svals.ctypes.data_as(N.p_f64), svals.shape[1])
    return args, bufs, ranks, svals


def _sweep_out(bufs, ranks, svals, dims, bonds, sites):
    """(cores, ranks, singular values) of the first ``sites`` cores and ``bonds`` bonds of a sweep, cut from its buffers;
    a core smaller than its buffer is copied so that the buffer is freed."""
    ranks = [int(r) for r in ranks][:bonds]
    cores = []
    for i in range(sites):
        shp = core_shape(i, len(dims), dims, ranks)
        core = bufs[i][:int(np.prod(shp, dtype=np.int64))].view(shp)
        cores.append(core if core.numel() == bufs[i].numel() else core.clone())
    return cores, ranks, [svals[i, :ranks[i]].copy() for i in range(bonds)]


def ttsvd(dense, dims, cutoff=1e-10, cutoff_mode="rsum2", max_bond=None, renorm=None):
    """Left-canonical MPS cores of ``dense`` (site order); returns (cores, ranks, svals)."""
    _dev(dense, "dense")
    dims = [int(d) for d in dims]
    args, bufs, ranks, svals = _sweep_args(dims, cutoff, cutoff_mode, renorm, max_bond, dense)
    N.check(N.load_library().ndmps_ttsvd(N.handle(), N.ptr(dense), N.dtype_code(dense.dtype), len(dims), N.i64_array(dims),
                                         *args), "ndmps_ttsvd")
    return _sweep_out(bufs, ranks, svals, dims, len(dims) - 1, len(dims))


class _DevicePointer:
    """Zero-copy torch view of library-owned device memory (``__cuda_array_interface__``)."""

    def __init__(self, ptr: int, count: int, typestr: str = "<f8"):
        self.__cuda_array_interface__ = {"shape": (int(count),), "typestr": typestr, "data": (int(ptr), False), "version": 2}


def ttsvd_sharded(dense_local, dims_local, world: int, allreduce=None, stop_bytes: int = 8 << 20, cutoff=1e-10,
                  cutoff_mode="rsum2", max_bond=None, renorm=None):
    """Sharded phase of the sweep on this rank's column block (``ndmps_ttsvd_sharded``).

    ``allreduce(tensor)`` must sum the float64 device tensor in place over the ranks (e.g.
    ``torch.distributed.all_reduce``); it is called once per Gram pass on the current stream.
    Returns (cores of the finished sites, their ranks, singular values, remainder[rows, cols])."""
    torch = _torch()
    _dev(dense_local, "dense_local")
    dims = [int(d) for d in dims_local]
    gdims = dims[:-1] + [dims[-1] * int(world)]
    args, bufs, ranks, svals = _sweep_args(gdims, cutoff, cutoff_mode, renorm, max_bond, dense_local)
    remainder = torch.empty(dense_local.numel(), dtype=dense_local.dtype, device=dense_local.device)
    sites_done = C.c_int(0)
    rshape = (C.c_int64 * 2)()
    failure = []

    def hook(_user, buf, count, _stream):
        try:
            allreduce(torch.as_tensor(_DevicePointer(buf, count), device=dense_local.device))
            return 0
        except Exception as exc:                     # never let an exception cross the C frame
            failure.append(exc)
            return 1

    cb = N.ALLREDUCE_FN(hook) if (world > 1 and allreduce is not None) else C.cast(None, N.ALLREDUCE_FN)
    if world > 1 and allreduce is None:
        raise ValueError("ttsvd_sharded: world > 1 needs an allreduce callable")
    rc = N.load_library().ndmps_ttsvd_sharded(
        N.handle(), N.ptr(dense_local), N.dtype_code(dense_local.dtype), len(dims), N.i64_array(dims), int(world), cb,
        None, int(stop_bytes), *args, C.byref(sites_done), N.ptr(remainder), remainder.numel(), rshape)
    if failure:
        raise failure[0]
    N.check(rc, "ndmps_ttsvd_sharded")
    done = sites_done.value
    cores, rk, sv = _sweep_out(bufs, ranks, svals, gdims, done, done)    # done < len(dims) - 1: never the last core
    rows, cols = int(rshape[0]), int(rshape[1])
    return cores, rk, sv, remainder[:rows * cols].view(rows, cols)


def interleave_shards(gathered, world: int, rows: int, cmid: int, dl: int):
    """gathered[g][r][c][t] (rank-major, as all-gathered) -> out[r][c][g][t] (site order)."""
    torch = _torch()
    _dev(gathered, "gathered")
    out = torch.empty(rows * cmid * world * dl, dtype=gathered.dtype, device=gathered.device)
    N.check(N.load_library().ndmps_interleave_shards(N.handle(), N.ptr(gathered), N.dtype_code(gathered.dtype), int(world),
                                                     int(rows), int(cmid), int(dl), N.ptr(out)), "ndmps_interleave_shards")
    return out.view(rows, cmid * world * dl)


def compress_bond(t1, t2, cutoff, cutoff_mode="rel", max_bond=None, renorm=0):
    """Truncate the bond between 2-D matricised cores t1 (a x r) and t2 (r x b)."""
    torch = _torch()
    _dev(t1), _dev(t2)
    a, r = int(t1.shape[0]), int(t1.shape[1])
    r2, b = int(t2.shape[0]), int(t2.shape[1])
    if r != r2 or t1.dtype != t2.dtype:
        raise ValueError("compress_bond: cores do not share the bond")
    o1 = torch.empty(a * r, dtype=t1.dtype, device=t1.device)
    o2 = torch.empty(r * b, dtype=t1.dtype, device=t1.device)
    n = C.c_int64(0)
    svals = np.zeros(r, dtype=np.float64)
    N.check(N.load_library().ndmps_compress_bond(N.handle(), N.ptr(t1), N.ptr(t2), N.dtype_code(t1.dtype), a, r, b,
                                                 float(cutoff), N.CUTOFF_MODES[cutoff_mode], int(max_bond or 0),
                                                 int(renorm), N.ptr(o1), N.ptr(o2), C.byref(n),
                                                 svals.ctypes.data_as(N.p_f64)), "ndmps_compress_bond")
    n = int(n.value)
    return o1[:a * n].clone().view(a, n), o2[:n * b].clone().view(n, b), svals[:n].copy()


def _ranks_of(cores):
    L = len(cores)
    if L == 1:
        return []
    return [int(cores[0].shape[1])] + [int(c.shape[2]) for c in cores[1:-1]]


def _dims_of(cores):
    if len(cores) == 1:
        return [int(cores[0].shape[0])]
    return [int(cores[0].shape[0])] + [int(c.shape[1]) for c in cores[1:]]


def _mps_args(cores):
    """(cores checked by ``_dev``, their pointer array, dtype code, ranks array): an MPS as the C ABI takes it."""
    cores = [_dev(c, "core") for c in cores]
    return cores, N.ptr_array(cores), N.dtype_code(cores[0].dtype), N.i64_array(_ranks_of(cores))


def contract_dense(cores):
    torch = _torch()
    cores, ptrs, code, ranks = _mps_args(cores)
    dims = _dims_of(cores)
    out = torch.empty(dims, dtype=cores[0].dtype, device=cores[0].device)
    N.check(N.load_library().ndmps_contract_dense(N.handle(), ptrs, code, len(cores), N.i64_array(dims), ranks, N.ptr(out)),
            "ndmps_contract_dense")
    return out


def region_box_axes(shape, index):
    """numpy basic indexing with step 1 -> (lo, hi, result shape, kept axes) of the box it selects in a volume of
    ``shape``; axis j of the result is volume axis ``kept[j]`` (an int drops its axis).

    ``index``: an int, a slice, ``Ellipsis`` or a tuple of them, with at most one ``Ellipsis`` and at most ``ndim``
    entries (missing trailing entries select whole axes).  Ints drop their axis and may be negative; slice bounds
    are clipped as numpy clips them.  Errors have numpy's types: ``IndexError`` for an int out of range, too many
    indices, a second ``Ellipsis`` or an index of another type, ``TypeError`` for a slice bound that is not an
    integer.  A slice step other than 1 (or None), ``None`` (new axis), booleans and arrays are not supported here
    and raise ``ValueError``."""
    import operator
    shape = tuple(int(s) for s in shape)
    ndim = len(shape)
    items = index if isinstance(index, tuple) else (index,)
    for it in items:
        if it is None or isinstance(it, (bool, np.bool_, np.ndarray, list)):
            raise ValueError(f"region index: {it!r} is not supported (ints, step-1 slices and Ellipsis only)")
        if not (it is Ellipsis or isinstance(it, slice) or hasattr(it, "__index__")):
            raise IndexError("only integers, slices (`:`) and ellipsis (`...`) are valid region indices")
    n_ell = sum(1 for it in items if it is Ellipsis)
    if n_ell > 1:
        raise IndexError("an index can only have a single ellipsis ('...')")
    if len(items) - n_ell > ndim:
        raise IndexError(f"too many indices: the volume is {ndim}-dimensional, but {len(items) - n_ell} were indexed")
    if n_ell:
        at = items.index(Ellipsis)
        items = items[:at] + (slice(None),) * (ndim - len(items) + 1) + items[at + 1:]
    items = items + (slice(None),) * (ndim - len(items))
    lo, hi, out_shape, kept = [], [], [], []
    for axis, (it, n) in enumerate(zip(items, shape)):
        if isinstance(it, slice):
            if it.step is not None and operator.index(it.step) != 1:
                raise ValueError(f"region index: slice step {it.step} on axis {axis} (only step 1 is supported)")
            start, stop, _ = slice(it.start, it.stop).indices(n)
            stop = max(stop, start)
            lo.append(start)
            hi.append(stop)
            out_shape.append(stop - start)
            kept.append(axis)
        else:
            i = operator.index(it)
            if not -n <= i < n:
                raise IndexError(f"index {i} is out of bounds for axis {axis} with size {n}")
            i += n if i < 0 else 0
            lo.append(i)
            hi.append(i + 1)
    return lo, hi, tuple(out_shape), tuple(kept)


def region_box(shape, index):
    """numpy basic indexing with step 1 -> (lo, hi, result shape) of the box it selects in a volume of ``shape``;
    ``region_box_axes`` without the kept axes."""
    return region_box_axes(shape, index)[:3]


def contract_region(cores, shape, lo, hi, plan=None):
    """Box [lo, hi) of the volume of ``shape`` that the cores encode, as a device tensor of shape hi - lo."""
    torch = _torch()
    cores, ptrs, code, ranks = _mps_args(cores)
    plan = plan or plan_for(tuple(shape))
    out = torch.empty([int(h) - int(l) for l, h in zip(lo, hi)], dtype=cores[0].dtype, device=cores[0].device)
    N.check(N.load_library().ndmps_contract_region(N.handle(), plan.handle, ptrs, code, ranks, N.i64_array(lo),
                                                   N.i64_array(hi), N.ptr(out)), "ndmps_contract_region")
    return out


PROJECTION_OPS = {"max": N.PROJ_MAX, "min": N.PROJ_MIN}


def project_region(cores, shape, lo, hi, axis, op, idct_last_axis: bool = False):
    """``op`` ("max" or "min", NaN propagating) over volume axis ``axis`` of the box [lo, hi) of the volume of ``shape``
    that the cores encode, as a device tensor of the box's shape without ``axis``."""
    torch = _torch()
    cores, ptrs, code, ranks = _mps_args(cores)
    plan = plan_for(tuple(shape))
    ext = [int(h) - int(l) for l, h in zip(lo, hi)]
    code_op = PROJECTION_OPS.get(op, 0)               # anything else: the library refuses it
    # a bad axis gets an empty output: the library refuses the axis before it looks at out
    out = torch.empty(ext[:axis] + ext[axis + 1:] if 0 <= axis < len(ext) else [0], dtype=cores[0].dtype,
                      device=cores[0].device)
    N.check(N.load_library().ndmps_project_region(N.handle(), plan.handle, ptrs, code, ranks, N.i64_array(lo),
                                                  N.i64_array(hi), int(axis), code_op, int(bool(idct_last_axis)),
                                                  N.ptr(out)), "ndmps_project_region")
    return out


def marginalize(cores, shape, levels):
    """Cores of the block mean of the volume of ``shape`` that ``cores`` encode, averaged over the finest ``levels``
    digits of each axis, in the layout of ``coarse_plan(shape, levels)``."""
    torch = _torch()
    cores, ptrs, code, ranks = _mps_args(cores)
    shape = tuple(int(s) for s in shape)
    ks = coarse_levels(shape, levels)
    cplan = coarse_plan(shape, ks)
    kept = _ranks_of(cores)[:cplan.levels - 1]
    shapes = [core_shape(i, cplan.levels, cplan.site_dims, kept) for i in range(cplan.levels)]
    out = [torch.empty(s, dtype=cores[0].dtype, device=cores[0].device) for s in shapes]
    N.check(N.load_library().ndmps_marginalize(N.handle(), plan_for(shape).handle, ptrs, code, ranks, N.i64_array(ks),
                                               N.ptr_array(out), N.i64_array([o.numel() for o in out])),
            "ndmps_marginalize")
    return out


def evaluate_points(cores, shape, coords, idct_last_axis: bool = False):
    """Values of the volume of ``shape`` at ``coords`` (int64 device tensor, K x ndim), as a device tensor of K values."""
    torch = _torch()
    cores, ptrs, code, ranks = _mps_args(cores)
    _dev(coords, "coords")
    if coords.dtype != torch.int64 or coords.ndim != 2 or coords.shape[1] != len(shape):
        raise ValueError("evaluate_points: coords must be an int64 (K, ndim) tensor")
    plan = plan_for(tuple(shape))
    count = int(coords.shape[0])
    out = torch.empty(count, dtype=cores[0].dtype, device=cores[0].device)
    N.check(N.load_library().ndmps_evaluate_points(N.handle(), plan.handle, ptrs, code, ranks, N.ptr(coords), count,
                                                   int(bool(idct_last_axis)), N.ptr(out)), "ndmps_evaluate_points")
    return out


def sample_points(cores, shape, coords, idct_last_axis: bool = False):
    """Multilinear interpolation of the volume of ``shape`` at ``coords`` (float64 device tensor, K x ndim), each
    coordinate clamped to [0, extent - 1]; a device tensor of K values.  A non-finite coordinate gives NaN."""
    torch = _torch()
    cores, ptrs, code, ranks = _mps_args(cores)
    _dev(coords, "coords")
    if coords.dtype != torch.float64 or coords.ndim != 2 or coords.shape[1] != len(shape):
        raise ValueError("sample_points: coords must be a float64 (K, ndim) tensor")
    plan = plan_for(tuple(shape))
    count = int(coords.shape[0])
    out = torch.empty(count, dtype=cores[0].dtype, device=cores[0].device)
    N.check(N.load_library().ndmps_sample_points(N.handle(), plan.handle, ptrs, code, ranks, N.ptr(coords), count,
                                                 int(bool(idct_last_axis)), N.ptr(out)), "ndmps_sample_points")
    return out


def grid_args(ndim, origin, steps, shape):
    """Validated (origin (ndim,), steps (m, ndim), shape (m,)) of an affine sampling grid, as float64 arrays and a tuple
    of ints.  ``origin`` and ``steps`` must be real and finite, 1 <= m <= 8, ``shape`` m non-negative ints; every
    coordinate of the grid must be finite too.  A wrong length, a non-real or non-finite value or a negative extent
    raises ``ValueError``; a bool or non-integer extent ``TypeError``."""
    import operator

    def real(a, what):
        a = np.asarray(a)
        if a.dtype == np.bool_ or a.dtype.kind not in "iuf":
            raise ValueError(f"{what} must be real numbers, got {a.dtype}")
        a = np.ascontiguousarray(a, dtype=np.float64)
        if not np.isfinite(a).all():
            raise ValueError(f"{what} must be finite")
        return a

    origin = real(origin, "origin")
    steps = real(steps, "steps")
    if origin.shape != (ndim,):
        raise ValueError(f"origin must have {ndim} values, got shape {origin.shape}")
    if steps.ndim != 2 or steps.shape[1] != ndim or not 1 <= steps.shape[0] <= 8:
        raise ValueError(f"steps must have shape (m, {ndim}) with 1 <= m <= 8, got {steps.shape}")
    out_shape = []
    for v in shape:
        if isinstance(v, (bool, np.bool_)) or not hasattr(v, "__index__"):
            raise TypeError(f"shape: {v!r} is not an integer")
        out_shape.append(operator.index(v))
    if len(out_shape) != steps.shape[0]:
        raise ValueError(f"shape has {len(out_shape)} extents for {steps.shape[0]} step vectors")
    if any(v < 0 for v in out_shape):
        raise ValueError(f"shape {tuple(out_shape)} has a negative extent")
    # the largest |coordinate| the grid reaches: finite, so is every coordinate
    with np.errstate(over="ignore"):
        far = np.abs(origin) + (np.maximum(np.array(out_shape, dtype=np.float64) - 1, 0)[:, None] * np.abs(steps)).sum(axis=0)
    if not np.isfinite(far).all():
        raise ValueError("the grid reaches a non-finite coordinate")
    return origin, steps, tuple(out_shape)


def sample_grid(cores, shape, origin, steps, out_shape, idct_last_axis: bool = False):
    """``sample_points`` at the affine grid origin + sum_j i_j steps[j] over ``out_shape`` (C order), with the
    coordinates computed in the kernel; a device tensor of ``out_shape``.  Arguments as ``grid_args`` returns them."""
    torch = _torch()
    cores, ptrs, code, ranks = _mps_args(cores)
    plan = plan_for(tuple(shape))
    origin = np.ascontiguousarray(origin, dtype=np.float64)
    steps = np.ascontiguousarray(steps, dtype=np.float64)
    out = torch.empty(tuple(int(v) for v in out_shape), dtype=cores[0].dtype, device=cores[0].device)
    N.check(N.load_library().ndmps_sample_grid(N.handle(), plan.handle, ptrs, code, ranks, origin.ctypes.data_as(N.p_f64),
                                               steps.ctypes.data_as(N.p_f64), N.i64_array(out_shape), len(out_shape),
                                               int(bool(idct_last_axis)), N.ptr(out)), "ndmps_sample_grid")
    return out


def overlap(cores_a, cores_b) -> float:
    cores_a, ptrs_a, code_a, ranks_a = _mps_args(cores_a)
    cores_b, ptrs_b, code_b, ranks_b = _mps_args(cores_b)
    dims = _dims_of(cores_a)
    if dims != _dims_of(cores_b):
        raise ValueError("overlap: the two MPS have different site dimensions")
    out = C.c_double()
    N.check(N.load_library().ndmps_overlap(N.handle(), ptrs_a, ranks_a, code_a, ptrs_b, ranks_b, code_b, len(cores_a),
                                           N.i64_array(dims), C.byref(out)), "ndmps_overlap")
    return out.value


# ---- K12 ---------------------------------------------------------------------------
def int_code(np_dtype) -> int:
    """The C ABI's name of an integer type: its bit count, negative when signed.  ValueError for anything
    ``np.iinfo`` rejects, as ``scale_to_dtype`` (``utils/filetools.py:26``) raises."""
    info = np.iinfo(np.dtype(np_dtype))            # ValueError for non-integer dtypes
    return int(info.bits) if info.min == 0 else -int(info.bits)


def _torch_int(code: int):
    torch = _torch()
    return {8: torch.uint8, 16: torch.uint16, 32: torch.uint32, 64: torch.uint64,
            -8: torch.int8, -16: torch.int16, -32: torch.int32, -64: torch.int64}[code]


def quantize(x, lo: float, hi: float, bits: int):
    """Min-max quantisation of a device tensor to the integer type `bits` names (8 / 16 / 32 / 64 unsigned, negative:
    signed) -- ``scale_to_dtype`` for every dtype ``np.iinfo`` knows."""
    torch = _torch()
    _dev(x)
    q = torch.empty(x.shape, dtype=_torch_int(int(bits)), device=x.device)
    N.check(N.load_library().ndmps_quantize(N.handle(), N.ptr(x), x.numel(), N.dtype_code(x.dtype), float(lo), float(hi),
                                            int(bits), N.ptr(q)), "ndmps_quantize")
    return q


def dequantize(q, lo: float, hi: float, bits: int, dtype):
    torch = _torch()
    _dev(q)
    x = torch.empty(q.shape, dtype=dtype, device=q.device)
    N.check(N.load_library().ndmps_dequantize(N.handle(), N.ptr(q), q.numel(), int(bits), float(lo), float(hi),
                                              N.dtype_code(dtype), N.ptr(x)), "ndmps_dequantize")
    return x


def to_host_int(q, np_dtype) -> np.ndarray:
    """Device integer tensor -> numpy array of `np_dtype` (bit reinterpretation where torch lacks numpy interop)."""
    np_dtype = np.dtype(np_dtype)
    try:
        out = q.cpu().numpy()
        if out.dtype == np_dtype:
            return out
    except (TypeError, RuntimeError):
        pass
    torch = _torch()
    raw = q.contiguous().view(torch.uint8).cpu().numpy()
    return raw.view(np_dtype).reshape(tuple(q.shape))


# ---- K9 ---------------------------------------------------------------------------
def ssim(a, b) -> float:
    _dev(a), _dev(b)
    out = C.c_double()
    N.check(N.load_library().ndmps_ssim(N.handle(), N.ptr(a), N.ptr(b), N.dtype_code(a.dtype), a.ndim,
                                        N.i64_array(a.shape), C.byref(out)), "ndmps_ssim")
    return out.value


def ssim_slices(a, b, axis: int) -> np.ndarray:
    _dev(a), _dev(b)
    out = np.empty(int(a.shape[axis]), dtype=np.float64)
    N.check(N.load_library().ndmps_ssim_slices(N.handle(), N.ptr(a), N.ptr(b), N.dtype_code(a.dtype),
                                               N.i64_array(a.shape), int(axis), out.ctypes.data_as(N.p_f64)),
            "ndmps_ssim_slices")
    return out


# ---- host-buffer end-to-end entry ---------------------------------------------------
def roundtrip_host(src: np.ndarray, max_bond=None, cutoff=1e-10, cutoff_mode="rsum2", renorm=None, out=None, extras=None):
    """NDMPS.from_tensor(src, max_bond=...).to_tensor() in ONE C-ABI call on host buffers
    (H2D, encode, sweep, boundary list + norm, contract, decode, D2H).  Returns (reconstruction, ranks);
    a dict passed as ``extras`` receives ``norm`` and ``boundary_list``."""
    if src.dtype not in (np.float32, np.float64):
        raise ValueError("roundtrip_host expects a float32 or float64 array")
    src = np.ascontiguousarray(src)
    plan = plan_for(tuple(src.shape))
    mode, renorm = _trim_mode(cutoff_mode, renorm)
    if out is None:
        out = np.empty_like(src)
    ranks = (C.c_int64 * max(plan.levels - 1, 1))()
    code = N.F32 if src.dtype == np.float32 else N.F64
    norm = C.c_double(0.0)
    bounds = np.zeros((plan.levels, 2), dtype=np.float64)
    N.check(N.load_library().ndmps_roundtrip_host(N.handle(), plan.handle, src.ctypes.data_as(C.c_void_p),
                                                  out.ctypes.data_as(C.c_void_p), code, float(cutoff), mode,
                                                  int(max_bond or 0), renorm, ranks, C.byref(norm),
                                                  bounds.ctypes.data_as(N.p_f64)), "ndmps_roundtrip_host")
    if extras is not None:
        extras["norm"] = norm.value
        extras["boundary_list"] = bounds
    return out, [int(r) for r in ranks][:plan.levels - 1]
