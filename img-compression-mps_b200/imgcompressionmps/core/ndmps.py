"""``NDMPS`` - the reference's class (``core/ndmps.py:11-277``) on the B200 device path.

Same constructor, methods, attribute names, argument meaning and error behaviour
as the reference; positional signatures are unchanged and the options the BASELINE
configs need are keyword-only with reference defaults:

* ``from_tensor(tensor, norm=False, mode="Std", *, max_bond=None, cutoff=1e-10,
  dtype=None, device=None)``  - quimb's ``from_dense(**split_opts)`` at
  ``core/ndmps.py:74`` already accepts ``max_bond`` / ``cutoff``; rule
  ``n = min(n_by_cutoff, max_bond)``.
* ``compress(cutoff, *, max_bond=None)`` - likewise for ``tensor_compress_bond``.

``dtype=None`` follows the input: float32 input stays float32 (the B200 fast path the
BASELINE configs name), everything else is promoted to float64 exactly as the
reference does at ``core/ndmps.py:56``.  Inputs may be numpy arrays (copied to the
device) or CUDA torch tensors (used in place, never aliased by the MPS).

Every numeric step is a call into ``libndmps_sm100.so``; there is no CPU path.
"""
from __future__ import annotations

import gzip
import io

import numpy as np

from .. import _ops
from ..utils.core import gen_encoding_map
from ..utils.filetools import get_num_bits
from .mps import DeviceMPS


def _torch():
    import torch
    return torch


def _to_device(tensor, dtype=None, device=None):
    """numpy / torch input -> contiguous CUDA tensor of the working dtype (always a copy
    or a fresh upload: the MPS never aliases the caller's data, as ``astype`` guarantees
    at ``core/ndmps.py:56``)."""
    torch = _torch()
    if isinstance(tensor, torch.Tensor):
        work = dtype or (torch.float32 if tensor.dtype == torch.float32 else torch.float64)
        dev = device or (tensor.device if tensor.is_cuda else torch.device("cuda"))
        return tensor.to(device=dev, dtype=work).contiguous()
    arr = np.asarray(tensor)
    work = dtype or (torch.float32 if arr.dtype == np.float32 else torch.float64)
    np_work = np.float32 if work == torch.float32 else np.float64
    host = np.ascontiguousarray(arr, dtype=np_work)
    return torch.from_numpy(host).to(device or "cuda", non_blocking=False)


def _coords_in(coords, ndim, name):
    """(K, ndim) point coordinates as a caller passes them: (the numpy array or CUDA tensor, whether it is a CUDA
    tensor, the function that turns a device result into the caller's form).  Anything but a numpy array (or what
    ``np.asarray`` takes) or a CUDA tensor, and a wrong shape, raise ``ValueError``."""
    torch = _torch()
    on_device = isinstance(coords, torch.Tensor)
    if on_device and not coords.is_cuda:
        raise ValueError(f"{name}: coords must be a numpy array or a CUDA tensor")
    if not on_device:
        coords = np.asarray(coords)
    if coords.ndim != 2 or int(coords.shape[1]) != ndim:
        raise ValueError(f"{name}: coords must have shape (K, {ndim}), got {tuple(coords.shape)}")
    return coords, on_device, (lambda out: out) if on_device else (lambda out: out.cpu().numpy())


class NDMPS:
    """Class for storing and compressing N-dimensional tensors using MPS (device-resident)."""

    def __init__(self, mps=None, qubit_size=None, encoding_map=None, boundary_list=None, norm: bool = True,
                 norm_value=None, mode: str = "Std", dim: int = None):
        self.qubit_size = qubit_size
        self._encoding_map = encoding_map
        self._shape = None
        self.mps = mps
        self.dim = dim
        self.norm = norm
        self.norm_value = norm_value
        self.mode = mode
        self.boundary_list = np.array(boundary_list)          # core/ndmps.py:34 (wraps None too)

    # The reference stores the (*shape, L) int64 map eagerly (8*L bytes per voxel, 9.7 GB at
    # 512^3).  Nothing on the device path needs it, so it is built on first access only.
    @property
    def encoding_map(self):
        if self._encoding_map is None and self._shape is not None:
            _, enc = gen_encoding_map(self._shape)
            self._encoding_map = np.moveaxis(enc, 0, -1)
        return self._encoding_map

    @encoding_map.setter
    def encoding_map(self, value):
        self._encoding_map = value

    @property
    def shape(self):
        return self._shape

    # ------------------------------------------------------------------ construction
    @classmethod
    def from_tensor(cls, tensor, norm: bool = False, mode: str = "Std", *, max_bond=None, cutoff: float = 1e-10,
                    dtype=None, device=None) -> "NDMPS":
        """N-D array -> MPS: (normalise) -> (DCT) -> site-order permutation -> TT-SVD
        (``core/ndmps.py:36-78``)."""
        vol = _to_device(tensor, dtype, device)
        shape = tuple(int(s) for s in vol.shape)
        plan = _ops.plan_for(shape)                      # raises ValueError like gen_encoding_map
        scale = 1.0
        if norm:
            scale = 1.0 / float(np.sqrt(_ops.sumsq(vol)))                 # core/ndmps.py:60-61
        if mode == "DCT":
            vol = _ops.dct_last_axis(vol, inverse=False)                  # core/ndmps.py:62-63
        dense = _ops.encode(vol, scale)                                   # core/ndmps.py:66-71
        del vol
        cores, _, svals = _ops.ttsvd(dense, plan.site_dims, cutoff=cutoff, cutoff_mode="rsum2",
                                     max_bond=max_bond)                  # core/ndmps.py:74
        del dense
        obj = cls(DeviceMPS(cores, plan.site_dims), np.array(plan.site_dims), None, None, norm, None, mode, len(shape))
        obj._shape = shape
        obj.singular_values = svals
        obj.update_boundary_list()                                        # core/ndmps.py:75
        obj.update_norm()                                                 # core/ndmps.py:76
        return obj

    # ------------------------------------------------------------------ bookkeeping
    def update_boundary_list(self):
        """Recompute min/max boundaries for each MPS tensor (``core/ndmps.py:80-82``)."""
        self.boundary_list = _ops.minmax(self.mps.cores)

    def update_norm(self):
        """Update stored norm of the current MPS (``core/ndmps.py:84-86``)."""
        self.norm_value = np.sqrt(self.mps @ self.mps)

    def compression_ratio(self):
        """MPS elements / original tensor elements (``core/ndmps.py:88-92``)."""
        return self.number_elements_in_MPS() / np.prod(self.qubit_size)

    def number_elements_in_MPS(self) -> int:
        return sum(t.size for t in self.mps)

    def bond_sizes(self):
        return self.mps.bond_sizes()

    def show(self):
        self.mps.show()

    # ------------------------------------------------------------------ truncation
    def compress(self, cutoff: float, *, max_bond=None):
        """Pairwise bond truncation, bonds left to right, relative cutoff, no
        canonicalisation in between (``core/ndmps.py:94-108``)."""
        cores = self.mps.cores
        L = len(cores)
        svals = []
        for i in range(1, L):
            t1, t2 = cores[i - 1], cores[i]
            a = t1.reshape(-1, t1.shape[-1])
            b = t2.reshape(t2.shape[0], -1)
            a_new, b_new, s = _ops.compress_bond(a, b, cutoff, "rel", max_bond)
            n = a_new.shape[1]
            cores[i - 1] = a_new.view(*t1.shape[:-1], n)
            cores[i] = b_new.view(n, *t2.shape[1:])
            svals.append(s)
        self.singular_values = svals
        self.update_boundary_list()
        self.update_norm()

    def continuous_compress(self, cutoff: float, print_ratio: bool = True):
        """20 compress steps with cutoffs linspace(0, 1, 20) * cutoff (``core/ndmps.py:110-125``)."""
        for c in np.linspace(0, 1, 20) * cutoff:
            self.compress(c)
            if print_ratio:
                print(f"Compression ratio at {c}: {self.compression_ratio()}")

    # ------------------------------------------------------------------ reconstruction
    @staticmethod
    def _decode_box(cores, plan, lo, hi, out_shape, last_axis=None):
        """Box [lo, hi) (lists) of the tensor ``cores`` encode in ``plan``'s layout as a CUDA tensor of ``out_shape``: K7
        for the whole tensor, else ``contract_region``.  ``last_axis`` (the inverse DCT or its block mean) maps whole
        lines, so the box is decoded over the full last axis, mapped and cropped to [lo[-1], hi[-1]) after."""
        shape = list(plan.shape)
        if last_axis is not None:
            crop = slice(lo[-1], hi[-1])
            lo, hi = lo[:-1] + [0], hi[:-1] + [shape[-1]]
        if lo == [0] * len(shape) and hi == shape:
            rec = _ops.decode(_ops.contract_dense(cores), shape, plan=plan)           # core/ndmps.py:140-148
        else:
            rec = _ops.contract_region(cores, shape, lo, hi, plan=plan)
        if last_axis is not None:
            rec = last_axis(rec)                                                      # core/ndmps.py:153
            rec = rec[..., crop].contiguous()
        return rec.view(out_shape)

    def to_tensor_device(self):
        """Reconstruction as a CUDA tensor of the original shape (no host copy): the box of the whole volume."""
        return self.to_tensor_region_device(())

    def to_tensor(self) -> np.ndarray:
        """MPS back to a numpy array (with inverse DCT in "DCT" mode); any other mode
        returns None as in the reference (``core/ndmps.py:131-153``)."""
        rec = self.to_tensor_device()
        return None if rec is None else rec.cpu().numpy()

    # ------------------------------------------------------------------ partial reconstruction (extension)
    def to_tensor_region_device(self, index):
        """``to_tensor_device()[index]`` for basic indexing with step 1 (ints, slices, ``...``; see
        ``_ops.region_box`` for the rules and errors), computed without the whole tensor: only the core slices the
        box touches are contracted, and the workspace is a small multiple of the box.  In "DCT" mode the inverse DCT
        runs along the whole last axis, so the box is decoded over the full last axis first and cropped after: that
        costs (last extent / box's last extent) times the memory and work of the box itself.  Any other mode returns
        None, as ``to_tensor`` does."""
        torch = _torch()
        lo, hi, out_shape = _ops.region_box(self._shape, index)
        if self.mode not in ("Std", "DCT"):
            return None
        cores = self.mps.cores
        if any(h == l for l, h in zip(lo, hi)):
            return torch.empty(out_shape, dtype=cores[0].dtype, device=cores[0].device)
        return self._decode_box(cores, _ops.plan_for(self._shape), lo, hi, out_shape,
                                (lambda x: _ops.dct_last_axis(x, inverse=True)) if self.mode == "DCT" else None)

    def to_tensor_region(self, index):
        """``to_tensor()[index]`` as a numpy array, without reconstructing the whole tensor (see
        ``to_tensor_region_device``); None for a mode other than "Std" / "DCT"."""
        rec = self.to_tensor_region_device(index)
        return None if rec is None else rec.cpu().numpy()

    def values_at(self, coords):
        """``to_tensor()[tuple(coords.T)]``: the values at K points, without reconstructing the whole tensor.

        ``coords``: integer array of shape (K, ndim), numpy (result: numpy array) or a CUDA tensor (result: CUDA
        tensor); negative coordinates count from the end, duplicates and K = 0 are allowed.  A coordinate outside
        [-extent, extent) raises ``IndexError``, a wrong shape ``ValueError``, a non-integer array ``IndexError``
        (numpy's errors for the same indexing).  Each point costs one bond-length dot product on the device; in "DCT"
        mode it costs one per element of its last-axis line (the inverse DCT of that line evaluated at the point).
        Any other mode returns None."""
        torch = _torch()
        coords, on_device, result = _coords_in(coords, len(self._shape), "values_at")
        integer = (not coords.dtype.is_floating_point and not coords.dtype.is_complex and coords.dtype != torch.bool
                   if on_device else np.issubdtype(coords.dtype, np.integer))
        if not integer:
            raise IndexError(f"values_at: coordinates must be integers, got {coords.dtype}")
        if on_device:
            coords = coords.to(torch.int64).contiguous()
            extent = torch.tensor(self._shape, dtype=torch.int64, device=coords.device)
            outside = bool(((coords < -extent) | (coords >= extent)).any().item()) if coords.numel() else False
        else:
            coords = np.ascontiguousarray(coords, dtype=np.int64)
            extent = np.array(self._shape, dtype=np.int64)
            outside = bool(((coords < -extent) | (coords >= extent)).any())
        if outside:
            raise IndexError(f"values_at: a coordinate is out of bounds for shape {self._shape}")
        if self.mode not in ("Std", "DCT"):
            return None
        cores = self.mps.cores
        dev = coords if on_device else torch.from_numpy(coords).to(cores[0].device)
        return result(_ops.evaluate_points(cores, self._shape, dev, idct_last_axis=self.mode == "DCT"))

    # ------------------------------------------------------------------ interpolated sampling (extension)
    def sample(self, coords):
        """``scipy.ndimage.map_coordinates(to_tensor(), coords.T, order=1, mode="nearest")``: the reconstruction
        linearly interpolated at K real-valued points, without reconstructing the whole tensor.

        ``coords``: real array of shape (K, ndim), numpy (result: numpy array) or a CUDA tensor (result: CUDA tensor),
        any real dtype; integer coordinates give ``values_at``'s values.  Each coordinate is clamped to
        [0, extent - 1] and the 2^ndim voxels around it are weighted multilinearly; duplicates and K = 0 are allowed.
        A wrong shape, a bool or non-real dtype, or a NaN / infinite coordinate raises ``ValueError``.  A sample costs
        up to 2^ndim bond-length dot products on the device (fewer where a coordinate is an integer); in "DCT" mode
        the inverse-DCT basis row is interpolated along the last axis, n * 2^(ndim-1) dot products per sample for a
        last extent n.  The path is for samples few compared with the voxels: oblique slices, probes along a path,
        a few in-between frames; the workspace is the decode chains and tables of ``values_at``, nothing of the
        size of the volume.  Any other mode returns None after the arguments are checked."""
        torch = _torch()
        coords, on_device, result = _coords_in(coords, len(self._shape), "sample")
        if on_device:
            real = not coords.dtype.is_complex and coords.dtype != torch.bool
        else:
            real = coords.dtype.kind in "iuf"
        if not real:
            raise ValueError(f"sample: coordinates must be real numbers, got {coords.dtype}")
        if on_device:
            coords = coords.to(torch.float64).contiguous()
            finite = bool(torch.isfinite(coords).all().item()) if coords.numel() else True
        else:
            coords = np.ascontiguousarray(coords, dtype=np.float64)
            finite = bool(np.isfinite(coords).all())
        if not finite:
            raise ValueError("sample: a coordinate is NaN or infinite")
        if self.mode not in ("Std", "DCT"):
            return None
        cores = self.mps.cores
        dev = coords if on_device else torch.from_numpy(coords).to(cores[0].device)
        return result(_ops.sample_points(cores, self._shape, dev, idct_last_axis=self.mode == "DCT"))

    def sample_grid_device(self, origin, steps, shape):
        """``sample`` at an affine grid, as a CUDA tensor of ``shape``: the value at index (i_0, .., i_{m-1}) is the
        sample at ``origin + sum_j i_j * steps[j]``.  The coordinates are computed on the device, so nothing of the
        output's size is allocated besides the output.

        ``origin``: ndim real numbers (voxel units, axis order of the volume); ``steps``: (m, ndim), 1 <= m <= 8;
        ``shape``: m non-negative ints.  Mismatched lengths, non-finite values and negative extents raise
        ``ValueError``.  For a volume of shape (D, H, W):

        * an oblique 512 x 512 plane through the centre c, spanned by orthonormal directions u and v (voxel units):
          ``origin = c - 255.5 * (u + v)``, ``steps = [u, v]``, ``shape = (512, 512)``;
        * a resample to (D', H', W') with the corners kept (``align_corners=True``):
          ``origin = (0, 0, 0)``, ``steps = diag((D - 1) / (D' - 1), (H - 1) / (H' - 1), (W - 1) / (W' - 1))``,
          ``shape = (D', H', W')``.

        Costs are ``sample``'s per output value.  Any other mode returns None after the arguments are checked."""
        torch = _torch()
        origin, steps, out_shape = _ops.grid_args(len(self._shape), origin, steps, shape)
        if self.mode not in ("Std", "DCT"):
            return None
        cores = self.mps.cores
        if 0 in out_shape:
            return torch.empty(out_shape, dtype=cores[0].dtype, device=cores[0].device)
        return _ops.sample_grid(cores, self._shape, origin, steps, out_shape, idct_last_axis=self.mode == "DCT")

    def sample_grid(self, origin, steps, shape):
        """``sample_grid_device(origin, steps, shape)`` as a numpy array; None for a mode other than "Std" / "DCT"."""
        rec = self.sample_grid_device(origin, steps, shape)
        return None if rec is None else rec.cpu().numpy()

    # ------------------------------------------------------------------ intensity projections (extension)
    def _projection_args(self, axis, op, index):
        """(lo, hi, volume axis, result shape) of ``project``; the argument errors of ``project_device``."""
        import operator
        if op not in _ops.PROJECTION_OPS:
            raise ValueError(f"project: op must be 'max' or 'min', got {op!r}")
        if isinstance(axis, (bool, np.bool_)) or not hasattr(axis, "__index__"):
            raise TypeError(f"project: axis {axis!r} is not an integer")
        axis = operator.index(axis)
        lo, hi, out_shape, kept = _ops.region_box_axes(self._shape, () if index is None else index)
        nd = len(out_shape)
        if not -nd <= axis < nd:
            raise ValueError(f"project: axis {axis} is out of bounds for an indexed result of {nd} dimensions")
        axis %= nd
        if out_shape[axis] == 0:
            raise ValueError(f"project: zero-size extent along axis {axis}, which has no {op}")
        return lo, hi, kept[axis], out_shape[:axis] + out_shape[axis + 1:]

    def project_device(self, axis, op: str = "max", index=None):
        """``getattr(np, op)(to_tensor()[index], axis=axis)`` as a CUDA tensor: a maximum (``op="max"``) or minimum
        (``"min"``) intensity projection, computed from the cores without holding the box in memory.

        ``index`` follows ``to_tensor_region``'s rules (ints, step-1 slices, ``...``; ``_ops.region_box``); None is the
        whole tensor, so ``project(0, index=(slice(100, 140),))`` is a 40-slice thick-slab MIP.  ``axis`` counts the
        axes of the indexed result and may be negative.  NaN propagates as in ``np.max`` / ``np.min``.  The result has
        the cores' dtype and the indexed shape without ``axis`` (0-d for a 1-D indexed result).  Every voxel of the box
        is still computed, but a block of at most 16 MB of the decode product at a time, each reduced into the result
        as soon as it is written; in "DCT" mode each block covers whole last-axis lines and is inverse-transformed
        first.  An ``op`` other than "max" / "min", an ``axis`` outside the indexed result's axes (a 0-d one has none)
        and an empty extent along ``axis`` raise ``ValueError``; index errors are ``region_box``'s.  An empty extent on
        another axis gives an empty result.  Any other mode returns None after the arguments are checked."""
        torch = _torch()
        lo, hi, vaxis, res_shape = self._projection_args(axis, op, index)
        if self.mode not in ("Std", "DCT"):
            return None
        cores = self.mps.cores
        if any(h == l for l, h in zip(lo, hi)):
            return torch.empty(res_shape, dtype=cores[0].dtype, device=cores[0].device)
        out = _ops.project_region(cores, self._shape, lo, hi, vaxis, op, idct_last_axis=self.mode == "DCT")
        return out.view(res_shape)

    def project(self, axis, op: str = "max", index=None):
        """``project_device(axis, op, index)`` as a numpy array; None for a mode other than "Std" / "DCT"."""
        rec = self.project_device(axis, op, index)
        return None if rec is None else rec.cpu().numpy()

    # ------------------------------------------------------------------ block-mean reconstruction (extension)
    def coarse_shape(self, levels) -> tuple:
        """Shape of ``to_tensor_coarse(levels)`` with no index: axis a averaged over its finest ``k_a`` digits, i.e.
        over blocks of ``b_a`` = the product of the axis' factors (``get_factorlist``) at the finest ``k_a`` levels.
        ``levels``: an int (every axis) or ``ndim`` ints, each in ``0 ..= L``; see ``_ops.coarse_levels`` for the
        errors.  Host only."""
        return _ops.coarse_plan(self._shape, levels).shape

    def to_tensor_coarse_device(self, levels, index=None):
        """``block_mean(to_tensor_device(), b)[index]``, the mean over non-overlapping blocks of ``b_a`` voxels along
        each axis (``coarse_shape`` gives the result's shape with no index), computed from the cores without the
        full-resolution tensor: each finest core is averaged over its digits and the trailing fully averaged sites
        fold into a boundary vector, then the reduced MPS is decoded like ``to_tensor`` (or like
        ``to_tensor_region`` for an ``index``, whose rules are ``_ops.region_box``'s, on the coarse shape).  In "DCT"
        mode every axis but the last is averaged in the cores and the last one through a block-averaged inverse DCT
        of its full lines.  Any other mode returns None after the arguments are checked."""
        torch = _torch()
        ks = _ops.coarse_levels(self._shape, levels)
        cplan = _ops.coarse_plan(self._shape, ks)
        cshape = cplan.shape
        lo, hi, out_shape = _ops.region_box(cshape, () if index is None else index)
        if self.mode not in ("Std", "DCT"):
            return None
        cores = self.mps.cores
        if any(h == l for l, h in zip(lo, hi)):
            return torch.empty(out_shape, dtype=cores[0].dtype, device=cores[0].device)
        if self.mode == "Std":
            return self._decode_box(_ops.marginalize(cores, self._shape, ks), cplan, lo, hi, out_shape)
        dks = ks[:-1] + (0,)                     # the last axis holds DCT coefficients: averaged after the inverse
        block = self._shape[-1] // cshape[-1]
        return self._decode_box(_ops.marginalize(cores, self._shape, dks), _ops.coarse_plan(self._shape, dks), lo, hi,
                                out_shape, lambda x: _ops.idct_block_mean_last_axis(x, block))

    def to_tensor_coarse(self, levels, index=None):
        """``to_tensor_coarse_device(levels, index)`` as a numpy array; None for a mode other than "Std" / "DCT"."""
        rec = self.to_tensor_coarse_device(levels, index)
        return None if rec is None else rec.cpu().numpy()

    # ------------------------------------------------------------------ core access
    def replace_tensordata(self, tensorlist):
        """Shape-asserting in-place overwrite of every core (``core/ndmps.py:163-175``)."""
        arrays = self.mps.arrays
        for i in range(len(arrays)):
            assert arrays[i].shape == tuple(tensorlist[i].shape)
            arrays[i][:] = tensorlist[i]
        self.update_boundary_list()
        self.update_norm()

    def return_tensors_data(self):
        return [t for t in self.mps.arrays]

    # ------------------------------------------------------------------ quantisation / size
    def _quantised_device(self, dtype):
        """[uint core on device], following scale_to_dtype (``filetools.py:20-26``) with each
        core's own current min/max."""
        code = _ops.int_code(dtype)              # any np.iinfo dtype, like the reference; ValueError otherwise
        bounds = _ops.minmax(self.mps.cores)
        return [_ops.quantize(c, lo, hi, code) for c, (lo, hi) in zip(self.mps.cores, bounds)], code

    def compress_to_dtype(self, dtype=np.uint16, replace: bool = False):
        """Integer-truncate each core (``core/ndmps.py:182-207``).  De-quantisation uses the
        STORED ``boundary_list`` like the reference (stale if cores were edited by hand)."""
        q_dev, bits = self._quantised_device(dtype)
        if replace:
            scaled_back = [_ops.dequantize(q, float(b[0]), float(b[1]), bits, c.dtype)
                           for q, b, c in zip(q_dev, self.boundary_list, self.mps.cores)]
            self.replace_tensordata(scaled_back)
        return [_ops.to_host_int(q, dtype) for q in q_dev]

    def get_bytesize_on_disk(self, dtype=np.uint16, replace: bool = False) -> int:
        """Sum of gzip sizes of the quantised cores (``core/ndmps.py:209-234``); the deflate
        runs on the host as in the reference."""
        total_bytes = 0
        for arr in self.compress_to_dtype(dtype, replace):
            buf = io.BytesIO()
            with gzip.GzipFile(fileobj=buf, mode="wb") as gz:
                gz.write(arr.tobytes())
            total_bytes += len(buf.getvalue())
        return total_bytes

    def compression_ratio_on_disk(self, dtype=np.uint16, replace: bool = False) -> float:
        original_size = np.prod(self.qubit_size) * get_num_bits(dtype) / 8.0
        return self.get_bytesize_on_disk(dtype, replace) / original_size

    def get_storage_space(self, dtype=np.uint16, verbose: bool = False) -> float:
        size_bytes = self.number_elements_in_MPS() * get_num_bits(dtype) / 8
        if verbose:
            print(f"The storage space is approximately: {size_bytes / 1024:.2f} KB")
        return size_bytes
