"""ctypes binding of ``libndmps_sm100.so`` (the C ABI declared in ``include/ndmps.h``).

There is deliberately no fallback: if the library is missing, or no sm_100 device
is present, every compute entry point raises.  PyTorch is used only for device
memory and streams; every kernel that runs is this library's.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from pathlib import Path

import numpy as np

F32, F64 = 0, 1
CUT_ABS, CUT_REL, CUT_SUM2, CUT_RSUM2, CUT_SUM1, CUT_RSUM1 = 1, 2, 3, 4, 5, 6
PROJ_MAX, PROJ_MIN = 1, 2
CUTOFF_MODES = {"abs": CUT_ABS, "rel": CUT_REL, "sum2": CUT_SUM2, "rsum2": CUT_RSUM2, "sum1": CUT_SUM1,
                "rsum1": CUT_RSUM1}

_LIB_NAME = "libndmps_sm100.so"
_lib = None
_lib_lock = threading.Lock()
_tls = threading.local()

i64, f64, vp, ci = C.c_int64, C.c_double, C.c_void_p, C.c_int
p_i64, p_f64, p_vp = C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_void_p)
# int (*ndmps_allreduce_fn)(void* user, double* buf_dev, int64_t count, void* stream)
ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p)

# name -> (restype, argtypes); kept in one table so the symbol test can walk it
PROTOTYPES = {
    "ndmps_version": (ci, []),
    "ndmps_last_error": (C.c_char_p, []),
    "ndmps_ctx_create": (ci, [p_vp]),
    "ndmps_ctx_destroy": (ci, [vp]),
    "ndmps_ctx_set_stream": (ci, [vp, vp]),
    "ndmps_ctx_sync": (ci, [vp]),
    "ndmps_ctx_launch_count": (i64, [vp]),
    "ndmps_ctx_set_option": (ci, [vp, C.c_char_p, i64]),
    "ndmps_ctx_get_stat": (ci, [vp, C.c_char_p, p_f64, ci]),
    "ndmps_ctx_profile": (ci, [vp, ci]),
    "ndmps_stage_count": (ci, []),
    "ndmps_stage_name": (C.c_char_p, [ci]),
    "ndmps_ctx_stage_times": (ci, [vp, p_f64, p_i64, ci]),
    "ndmps_plan_create": (ci, [ci, p_i64, ci, p_i64, p_vp]),
    "ndmps_plan_destroy": (ci, [vp]),
    "ndmps_plan_site_dims": (ci, [vp, p_i64]),
    "ndmps_plan_layout": (ci, [vp, C.POINTER(ci), C.POINTER(ci), p_i64, p_i64]),
    "ndmps_plan_coarse": (ci, [vp, p_i64, p_vp]),
    "ndmps_plan_debug_offsets": (ci, [vp, ci, i64, i64, p_i64]),
    "ndmps_plan_debug_tile_info": (ci, [vp, ci, p_i64]),
    "ndmps_plan_debug_apply_tiled": (ci, [vp, ci, vp, vp]),
    "ndmps_plan_debug_bit_info": (ci, [vp, ci, p_i64]),
    "ndmps_plan_debug_apply_bits": (ci, [vp, ci, vp, vp]),
    "ndmps_encode": (ci, [vp, vp, vp, vp, ci, f64]),
    "ndmps_decode": (ci, [vp, vp, vp, vp, ci]),
    "ndmps_sumsq": (ci, [vp, vp, i64, ci, p_f64]),
    "ndmps_minmax": (ci, [vp, p_vp, p_i64, ci, ci, p_f64]),
    "ndmps_psnr_terms": (ci, [vp, vp, vp, i64, ci, p_f64]),
    "ndmps_dct_last_axis": (ci, [vp, vp, vp, i64, i64, ci, ci]),
    "ndmps_idct_block_mean_last_axis": (ci, [vp, vp, vp, i64, i64, i64, ci]),
    "ndmps_gram": (ci, [vp, vp, i64, i64, i64, ci, ci, vp]),
    "ndmps_eigh": (ci, [vp, vp, i64, vp, vp, C.POINTER(ci)]),
    "ndmps_eigh_topk": (ci, [vp, vp, i64, i64, vp, vp]),
    "ndmps_ttsvd_sharded": (ci, [vp, vp, ci, ci, p_i64, ci, ALLREDUCE_FN, vp, i64, f64, ci, i64, ci,
                                p_vp, p_i64, p_i64, p_f64, i64, C.POINTER(ci), vp, i64, p_i64]),
    "ndmps_interleave_shards": (ci, [vp, vp, ci, ci, i64, i64, i64, vp]),
    "ndmps_gemm": (ci, [vp, i64, i64, i64, f64, vp, ci, i64, i64, vp, ci, i64, i64, vp, ci, i64]),
    "ndmps_ttsvd": (ci, [vp, vp, ci, ci, p_i64, f64, ci, i64, ci, p_vp, p_i64, p_i64, p_f64, i64]),
    "ndmps_compress_bond": (ci, [vp, vp, vp, ci, i64, i64, i64, f64, ci, i64, ci, vp, vp, p_i64, p_f64]),
    "ndmps_contract_dense": (ci, [vp, p_vp, ci, ci, p_i64, p_i64, vp]),
    "ndmps_contract_region": (ci, [vp, vp, p_vp, ci, p_i64, p_i64, p_i64, vp]),
    "ndmps_evaluate_points": (ci, [vp, vp, p_vp, ci, p_i64, vp, i64, ci, vp]),
    "ndmps_sample_points": (ci, [vp, vp, p_vp, ci, p_i64, vp, i64, ci, vp]),
    "ndmps_sample_grid": (ci, [vp, vp, p_vp, ci, p_i64, p_f64, p_f64, p_i64, ci, ci, vp]),
    "ndmps_region_debug_offsets": (ci, [vp, p_i64, p_i64, p_i64, p_i64]),
    "ndmps_project_region": (ci, [vp, vp, p_vp, ci, p_i64, p_i64, p_i64, ci, ci, ci, vp]),
    "ndmps_project_debug_offsets": (ci, [vp, p_i64, p_i64, ci, i64, p_i64, p_i64]),
    "ndmps_marginalize": (ci, [vp, vp, p_vp, ci, p_i64, p_i64, p_vp, p_i64]),
    "ndmps_overlap": (ci, [vp, p_vp, p_i64, ci, p_vp, p_i64, ci, ci, p_i64, p_f64]),
    "ndmps_quantize": (ci, [vp, vp, i64, ci, f64, f64, ci, vp]),
    "ndmps_dequantize": (ci, [vp, vp, i64, ci, f64, f64, ci, vp]),
    "ndmps_ssim": (ci, [vp, vp, vp, ci, ci, p_i64, p_f64]),
    "ndmps_ssim_slices": (ci, [vp, vp, vp, ci, p_i64, ci, p_f64]),
    "ndmps_roundtrip_host": (ci, [vp, vp, vp, vp, ci, f64, ci, i64, ci, p_i64, p_f64, p_f64]),
}


class NativeError(RuntimeError):
    pass


def library_path() -> Path:
    override = os.environ.get("NDMPS_LIBRARY")
    return Path(override) if override else Path(__file__).resolve().parent / _LIB_NAME


def load_library():
    """dlopen the C-ABI library and attach prototypes.  Needs no GPU."""
    global _lib
    if _lib is not None:
        return _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        path = library_path()
        if not path.exists():
            raise NativeError(
                f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C img-compression-mps_b200/csrc`). There is no CPU fallback.")
        lib = C.CDLL(str(path))
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str = ""):
    if rc == 0:
        return
    msg = load_library().ndmps_last_error().decode("utf-8", "replace")
    if rc == -1:
        raise ValueError(msg or what)
    raise NativeError(f"{what} failed ({rc}): {msg}")


class Context:
    """One ndmps_ctx (device workspace + stream) per host thread and device."""

    def __init__(self):
        import torch
        if not torch.cuda.is_available():
            raise NativeError("imgcompressionmps needs a CUDA device (B200, sm_100a); none is visible. "
                              "There is no CPU fallback.")
        self.lib = load_library()
        self.device = torch.cuda.current_device()
        handle = vp()
        check(self.lib.ndmps_ctx_create(C.byref(handle)), "ndmps_ctx_create")
        self.handle = handle
        for key, val in os.environ.items():
            if key.startswith("NDMPS_OPT_"):
                self.set_option(key[len("NDMPS_OPT_"):].lower(), int(val))

    def bind_stream(self):
        import torch
        stream = torch.cuda.current_stream().cuda_stream
        check(self.lib.ndmps_ctx_set_stream(self.handle, vp(stream)), "ndmps_ctx_set_stream")
        return self.handle

    def set_option(self, name: str, value: int):
        check(self.lib.ndmps_ctx_set_option(self.handle, name.encode(), int(value)), "ndmps_ctx_set_option")

    def stat(self, name: str, reset: bool = False) -> float:
        out = C.c_double()
        check(self.lib.ndmps_ctx_get_stat(self.handle, name.encode(), C.byref(out), int(bool(reset))), "ndmps_ctx_get_stat")
        return out.value

    def profile(self, enable: bool):
        check(self.lib.ndmps_ctx_profile(self.handle, int(bool(enable))), "ndmps_ctx_profile")

    def stage_times(self, reset: bool = True) -> dict:
        """{stage: (ms, calls)} accumulated since the last reset (device time, CUDA events)."""
        n = self.lib.ndmps_stage_count()
        ms = (C.c_double * n)()
        calls = (C.c_int64 * n)()
        check(self.lib.ndmps_ctx_stage_times(self.handle, ms, calls, int(bool(reset))), "ndmps_ctx_stage_times")
        return {self.lib.ndmps_stage_name(i).decode(): (ms[i], int(calls[i])) for i in range(n)}

    def launch_count(self) -> int:
        return int(self.lib.ndmps_ctx_launch_count(self.handle))

    def __del__(self):
        try:
            if getattr(self, "handle", None) and self.lib is not None:
                self.lib.ndmps_ctx_destroy(self.handle)
        except Exception:
            pass


def context() -> Context:
    import torch
    dev = torch.cuda.current_device() if torch.cuda.is_available() else -1
    table = getattr(_tls, "ctx", None)
    if table is None:
        table = _tls.ctx = {}
    if dev not in table:
        table[dev] = Context()
    return table[dev]


def handle():
    """Context handle bound to torch's current stream."""
    return context().bind_stream()


# ---- small marshalling helpers ---------------------------------------------------
def dtype_code(torch_dtype) -> int:
    import torch
    if torch_dtype == torch.float32:
        return F32
    if torch_dtype == torch.float64:
        return F64
    raise ValueError(f"Unsupported dtype {torch_dtype!r}: the device path computes in float32 or float64")


def i64_array(values):
    values = [int(v) for v in values]
    return (C.c_int64 * max(len(values), 1))(*values)


def ptr_array(tensors):
    return (C.c_void_p * max(len(tensors), 1))(*[t.data_ptr() for t in tensors])


def ptr(t):
    return vp(t.data_ptr())


class Plan:
    """Permutation plan for one volume shape (ndmps_plan); needs no GPU to build."""

    def __init__(self, shape, factors: np.ndarray):
        self.lib = load_library()
        self.shape = tuple(int(s) for s in shape)
        factors = np.ascontiguousarray(factors, dtype=np.int64)
        self.levels, ndim = factors.shape
        assert ndim == len(self.shape)
        h = vp()
        check(self.lib.ndmps_plan_create(ndim, i64_array(self.shape), int(self.levels),
                                         factors.ctypes.data_as(p_i64), C.byref(h)), "ndmps_plan_create")
        self._adopt(h, factors)

    def _adopt(self, h, factors):
        self.handle = h
        self.factors = factors
        dims = (C.c_int64 * self.levels)()
        check(self.lib.ndmps_plan_site_dims(h, dims), "ndmps_plan_site_dims")
        self.site_dims = [int(d) for d in dims]
        self.total = int(np.prod(self.shape, dtype=np.int64)) if len(self.shape) else 0

    def coarse(self, drop_levels) -> "Plan":
        """Plan of the block-mean tensor that averages the finest ``drop_levels[a]`` digits of axis a
        (``ndmps_plan_coarse`` decides its shape and factor table; this only reads them back)."""
        h = vp()
        check(self.lib.ndmps_plan_coarse(self.handle, i64_array(drop_levels), C.byref(h)), "ndmps_plan_coarse")
        out = Plan.__new__(Plan)
        out.lib = self.lib
        out.handle = h                                   # freed by __del__ even if a read below fails
        ndim, levels = C.c_int(), C.c_int()
        check(self.lib.ndmps_plan_layout(h, C.byref(ndim), C.byref(levels), None, None), "ndmps_plan_layout")
        shape = np.empty(ndim.value, dtype=np.int64)
        factors = np.empty((levels.value, ndim.value), dtype=np.int64)
        check(self.lib.ndmps_plan_layout(h, C.byref(ndim), C.byref(levels), shape.ctypes.data_as(p_i64),
                                         factors.ctypes.data_as(p_i64)), "ndmps_plan_layout")
        out.shape = tuple(int(s) for s in shape)
        out.levels = levels.value
        out._adopt(h, factors)
        return out

    def debug_offsets(self, inverse: bool, first: int, count: int) -> np.ndarray:
        out = np.empty(count, dtype=np.int64)
        check(self.lib.ndmps_plan_debug_offsets(self.handle, int(bool(inverse)), int(first), int(count),
                                                out.ctypes.data_as(p_i64)), "ndmps_plan_debug_offsets")
        return out

    def region_debug(self, lo, hi):
        """(dict(s, rows, cols), flat site-order index per voxel of the box [lo, hi)) as the region path computes it."""
        count = int(np.prod([int(h) - int(l) for l, h in zip(lo, hi)], dtype=np.int64)) if len(lo) else 0
        out = np.empty(max(count, 0), dtype=np.int64)
        info = (C.c_int64 * 3)()
        check(self.lib.ndmps_region_debug_offsets(self.handle, i64_array(lo), i64_array(hi), info,
                                                  out.ctypes.data_as(p_i64)), "ndmps_region_debug_offsets")
        return dict(zip(("s", "rows", "cols"), (int(v) for v in info))), out

    def project_debug(self, lo, hi, axis: int, block_elems: int):
        """(dict(s, rows, cols, blocks), site-order index read, block that reads it), both (output elements, extent along
        ``axis``), as the projection of the box [lo, hi) along ``axis`` computes them with blocks of at most
        ``block_elems`` elements of T (at least one axis-0 high part each)."""
        ext = [int(h) - int(l) for l, h in zip(lo, hi)]
        e = ext[axis] if 0 <= axis < len(ext) else 0
        count = int(np.prod([x for a, x in enumerate(ext) if a != axis], dtype=np.int64))
        out = np.empty((2, max(count, 0), max(e, 0)), dtype=np.int64)
        info = (C.c_int64 * 4)()
        check(self.lib.ndmps_project_debug_offsets(self.handle, i64_array(lo), i64_array(hi), int(axis), int(block_elems),
                                                   info, out.ctypes.data_as(p_i64)), "ndmps_project_debug_offsets")
        return dict(zip(("s", "rows", "cols", "blocks"), (int(v) for v in info))), out[0], out[1]

    def tile_info(self, inverse: bool) -> dict:
        out = (C.c_int64 * 6)()
        check(self.lib.ndmps_plan_debug_tile_info(self.handle, int(bool(inverse)), out), "ndmps_plan_debug_tile_info")
        return dict(zip(("tiled", "tile", "dst_run", "src_run", "tiles", "bank_conflict"), (int(v) for v in out)))

    def apply_tiled_host(self, inverse: bool, src: np.ndarray) -> np.ndarray:
        src = np.ascontiguousarray(src, dtype=np.int32).reshape(-1)
        dst = np.full(src.shape, -1, dtype=np.int32)
        check(self.lib.ndmps_plan_debug_apply_tiled(self.handle, int(bool(inverse)), src.ctypes.data_as(C.c_void_p),
                                                    dst.ctypes.data_as(C.c_void_p)), "ndmps_plan_debug_apply_tiled")
        return dst

    def bit_info(self, inverse: bool) -> dict:
        out = (C.c_int64 * 7)()
        check(self.lib.ndmps_plan_debug_bit_info(self.handle, int(bool(inverse)), out), "ndmps_plan_debug_bit_info")
        return dict(zip(("bits", "nbits", "row_shift", "pair_shift", "ctas", "dst_run", "src_run"), (int(v) for v in out)))

    def apply_bits_host(self, inverse: bool, src: np.ndarray) -> np.ndarray:
        src = np.ascontiguousarray(src, dtype=np.int32).reshape(-1)
        dst = np.full(src.shape, -1, dtype=np.int32)
        check(self.lib.ndmps_plan_debug_apply_bits(self.handle, int(bool(inverse)), src.ctypes.data_as(C.c_void_p),
                                                   dst.ctypes.data_as(C.c_void_p)), "ndmps_plan_debug_apply_bits")
        return dst

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.ndmps_plan_destroy(self.handle)
        except Exception:
            pass
