"""Every kernel the GEMM, Gram, DCT, reduction and quantisation entry points dispatch to, on both sides of each selection
rule, against plain float64 numpy references on the same seeded inputs.

The entry points pick a kernel from the shape, the dtypes, the strides, the pointer alignment and the SM count.  Each
case below names the kernel it is meant to reach, and a ``torch.profiler`` trace of the call asserts that this kernel
ran (and that the competing ones did not): if a threshold moves, the case fails instead of quietly testing another
kernel.  Shapes on either side of the output-tile rule are derived from the device's SM count.

Products are checked element by element, not against the largest entry (u = 2^-53):

* float64 output: ``|got - ref| <= 4 k u (|A| |B|)_ij``, ref the float64 numpy product;
* float32 output: the same plus ``2^-24 |ref|_ij``: the float64 result rounded once;
* tcgen05 (bf16x3 planes): 1e-6 of the largest entry, the path's documented accuracy.

A float32 accumulation, a float32 rounding of a float64 output or a second rounding misses these by orders of
magnitude."""
import contextlib
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
scipy_fft = pytest.importorskip("scipy.fft")

from oracle import quantise as OQ          # noqa: E402

U = 2.0 ** -53
F32, F64 = torch.float32, torch.float64
CNAME = {F32: "float", F64: "double"}       # template arguments as the demangled kernel names spell them
NP = {F32: np.float32, F64: np.float64}


@pytest.fixture(scope="module")
def lib():
    from imgcompressionmps import _native, _ops
    return _native, _ops


@pytest.fixture()
def ctx(lib):
    native, _ = lib
    c = native.context()
    yield c
    for name, value in (("gram_path", 0), ("gemm_path", 0), ("gemm_out_t", 0), ("tc", 1), ("tc_waves", 1)):
        c.set_option(name, value)


@pytest.fixture(scope="module")
def sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


@contextlib.contextmanager
def kernels():
    """Names of the CUDA kernels launched inside the block; filled when the block ends."""
    names = []
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        yield names
        torch.cuda.synchronize()
    names.extend(sorted({e.name for e in prof.events()}))


def assert_ran(names, want, absent=()):
    for w in [want] if isinstance(want, str) else want:
        assert any(w in n for n in names), f"{w} did not run; kernels: {names}"
    for a in absent:
        assert not any(a in n for n in names), f"{a} ran; kernels: {names}"


def assert_product(got, ref, mag, k, out_dtype):
    """Per-element bound of a float64 accumulation (see the module docstring); NaN fails."""
    got = got.double().cpu().numpy() if isinstance(got, torch.Tensor) else got
    bound = 4.0 * k * U * mag
    if out_dtype == F32:
        bound = bound + 2.0 ** -24 * np.abs(ref)
    err = np.abs(got - ref)
    bad = ~(err <= bound)
    assert not bad.any(), (f"{int(bad.sum())} of {bad.size} elements out of bound; worst error / bound = "
                           f"{float(np.nanmax(err / np.maximum(bound, 1e-300)))}")


def rounded(rng, shape, dtype):
    """Standard normal float64 values, rounded to `dtype` (so the float64 copy is what the kernel reads)."""
    return rng.standard_normal(shape).astype(NP[dtype]).astype(np.float64)


def dev(x, dtype):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=NP[dtype])).cuda()


# ---- GEMM ------------------------------------------------------------------------------------------------------
# gemm_dmma_kernel takes a product when A is K-contiguous, B N-contiguous, m >= 48, n >= 64, k >= 4 and there are at
# least sm_count 64 x 128 output tiles (gemm_dmma.cu); its tile height is 64 when m <= 64 or m % 128 is in 1..64 with
# m < 512, else 128.  Everything else runs gemm_f64acc_kernel (SIMT), with split-K (splitk_reduce_kernel) when it has
# fewer than 2 sm_count 64 x 64 tiles and k >= 128.
#   id: ((m, n, k) from the SM count, alpha, A stored K-strided, B stored K-major, ldc - n, route of the default dispatch)
GEMM_CASES = {
    "projection-64x32768x512": (lambda sm: (64, 32768, 512), 1.0, False, False, 0, "dmma64"),
    "m192-ragged-n-k17": (lambda sm: (192, 128 * -(-sm // 3) - 37, 17), -0.375, False, False, 0, "dmma64"),
    "m192-ldc-padded": (lambda sm: (192, 128 * -(-sm // 3) - 37, 17), 1.0, False, False, 5, "dmma64"),
    "m448-below-512": (lambda sm: (448, 128 * -(-sm // 7), 40), 1.0, False, False, 0, "dmma64"),
    "m48": (lambda sm: (48, 128 * sm, 33), 1.0, False, False, 0, "dmma64"),
    "tiles=sm": (lambda sm: (64, 128 * sm, 256), 1.0, False, False, 0, "dmma64"),
    "m65": (lambda sm: (65, 128 * -(-sm // 2), 20), 1.0, False, False, 0, "dmma128"),
    "m200-last-tile-1-col-k1000": (lambda sm: (200, 128 * (-(-sm // 4) - 1) + 1, 1000), 1.0, False, False, 0, "dmma128"),
    "m576-odd-n-k4": (lambda sm: (576, 128 * -(-sm // 9) - 1, 4), -0.375, False, False, 0, "dmma128"),
    "reconstruction-4096x4096x64": (lambda sm: (4096, 4096, 64), 1.0, False, False, 0, "dmma128"),
    "n64": (lambda sm: (64 * sm, 64, 8), 1.0, False, False, 0, "dmma128"),
    "tiles=sm-1-splitk": (lambda sm: (64, 128 * (sm - 1), 256), 1.0, False, False, 0, "simt+splitk"),
    "m47": (lambda sm: (47, 128 * sm, 33), 1.0, False, False, 0, "simt"),
    "n63": (lambda sm: (64 * sm, 63, 8), 1.0, False, False, 0, "simt"),
    "k3": (lambda sm: (64, 128 * sm, 3), 1.0, False, False, 0, "simt"),
    "A-K-strided": (lambda sm: (64, 128 * sm, 256), -0.375, True, False, 0, "simt"),
    "B-K-major": (lambda sm: (64, 128 * sm, 256), 1.0, False, True, 0, "simt"),
    "bond-sized-splitk-ldc-padded": (lambda sm: (65, 130, 1000), 1.0, False, False, 3, "simt+splitk"),
}
DTYPES3 = [(a, b, c) for a in (F32, F64) for b in (F32, F64) for c in (F32, F64)]


def _gemm_route(route, da, db, dc):
    """(kernels that must run, kernels that must not)"""
    simt = f"gemm_f64acc_kernel<{CNAME[da]}, {CNAME[db]}>"
    if route.startswith("dmma"):
        bm = route[4:]
        other = "128" if bm == "64" else "64"
        return ([f"gemm_dmma_kernel<{bm}, {CNAME[da]}, {CNAME[db]}, {CNAME[dc]}>"],
                ["gemm_f64acc_kernel", "splitk_reduce_kernel", f"gemm_dmma_kernel<{other},", "gemm_tc_kernel"])
    if route == "simt+splitk":
        return [simt, "splitk_reduce_kernel"], ["gemm_dmma_kernel", "gemm_tc_kernel"]
    return [simt], ["gemm_dmma_kernel", "splitk_reduce_kernel", "gemm_tc_kernel"]


def _gemm(lib, a, b, alpha, out_dtype, pad):
    """ops.gemm, or the C ABI directly when the output rows are padded (ldc = n + pad; the padding stays NaN)."""
    native, ops = lib
    if pad == 0:
        return ops.gemm(a, b, out_dtype=out_dtype, alpha=alpha), None
    (m, k), n = a.shape, b.shape[1]
    c = torch.full((m, n + pad), float("nan"), dtype=out_dtype, device="cuda")
    native.check(native.load_library().ndmps_gemm(
        native.handle(), m, n, k, float(alpha), native.ptr(a), native.dtype_code(a.dtype), a.stride(0), a.stride(1),
        native.ptr(b), native.dtype_code(b.dtype), b.stride(0), b.stride(1), native.ptr(c), native.dtype_code(out_dtype),
        n + pad), "ndmps_gemm")
    return c[:, :n], c[:, n:]


@pytest.mark.parametrize("dtypes", DTYPES3, ids=lambda d: "-".join("f32" if t == F32 else "f64" for t in d))
@pytest.mark.parametrize("case", list(GEMM_CASES), ids=str)
def test_gemm_routes(lib, ctx, sm, case, dtypes):
    """The default dispatch reaches the case's kernel, and gemm_path = 2 (SIMT) gives the same inputs within the same
    bound."""
    shape, alpha, a_kstrided, b_kmajor, pad, route = GEMM_CASES[case]
    m, n, k = shape(sm)
    da, db, dc = dtypes
    rng = np.random.default_rng([m, n, k])
    a64, b64 = rounded(rng, (m, k), da), rounded(rng, (k, n), db)
    a = dev(a64.T, da).t() if a_kstrided else dev(a64, da)
    b = dev(b64.T, db).t() if b_kmajor else dev(b64, db)
    ref = alpha * (a64 @ b64)
    mag = abs(alpha) * (np.abs(a64) @ np.abs(b64))
    for path, want in ((0, route), (2, "simt-any")):
        ctx.set_option("gemm_path", path)
        with kernels() as ran:
            got, padding = _gemm(lib, a, b, alpha, dc, pad)
        if want == "simt-any":
            assert_ran(ran, f"gemm_f64acc_kernel<{CNAME[da]}, {CNAME[db]}>", ["gemm_dmma_kernel", "gemm_tc_kernel"])
        else:
            assert_ran(ran, *_gemm_route(want, da, db, dc))
        assert_product(got, ref, mag, k, dc)
        if padding is not None:
            assert bool(torch.isnan(padding).all()), "a store landed in the padding of the output rows"


# ---- Gram ------------------------------------------------------------------------------------------------------
# gram_dmma_kernel (gram_dmma.cu) takes G = M M^T of a float32 M with 48 <= rows <= 4096, cols >= 128, ld % 4 == 0 and
# a 16-byte aligned base; everything else (float64, side = 1, the other shapes) is G through gemm_f64acc_kernel.
# The padding columns between cols and ld, and 64 elements past the end, hold NaN: any over-read shows in the result.
GRAM_ROWS = {47: "simt", 48: "dmma", 129: "dmma", 360: "dmma", 4096: "dmma", 4097: "simt"}
GRAM_COLS = {                     # id: (cols, ld, route)
    "cols127-ld128": (127, 128, "simt"),        # cols below 4 x BK
    "cols128": (128, 128, "dmma"),
    "cols1000": (1000, 1000, "dmma"),
    "cols1001-ld1004": (1001, 1004, "dmma"),    # K tail of one float in front of NaN padding
    "cols1001-ld1001": (1001, 1001, "simt"),    # ld % 4 != 0
}
#   id: (rows, cols, ld, dtype, side, offset of the base in elements, route)
GRAM_CASES = {f"rows{r}-{c}": (r, cols, ld, F32, 0, 0, "dmma" if rr == cr == "dmma" else "simt")
              for r, rr in GRAM_ROWS.items() for c, (cols, ld, cr) in GRAM_COLS.items()}
GRAM_CASES.update({
    "base+1-float": (360, 1000, 1000, F32, 0, 1, "simt"),      # 4-byte aligned base
    "base+4-floats": (360, 1000, 1000, F32, 0, 4, "dmma"),     # 16-byte aligned again
    "f64-side0": (360, 1001, 1004, F64, 0, 0, "simt"),
    "f64-side1": (360, 1001, 1004, F64, 1, 0, "simt"),
    "f32-side1": (360, 1001, 1004, F32, 1, 0, "simt"),
    "f32-side1-rows4097": (4097, 130, 132, F32, 1, 3, "simt"),
})


def _gram(lib, base, rows, cols, ld, dtype, side):
    native, _ = lib
    n = rows if side == 0 else cols
    g = torch.empty((n, n), dtype=F64, device="cuda")
    native.check(native.load_library().ndmps_gram(native.handle(), native.ptr(base), rows, cols, ld,
                                                  native.dtype_code(dtype), side, native.ptr(g)), "ndmps_gram")
    return g


@pytest.mark.parametrize("case", list(GRAM_CASES), ids=str)
def test_gram_routes(lib, ctx, case):
    rows, cols, ld, dtype, side, offset, route = GRAM_CASES[case]
    rng = np.random.default_rng([rows, cols, ld, side, offset])
    m64 = rounded(rng, (rows, cols), dtype)
    buf = torch.full((offset + rows * ld + 64,), float("nan"), dtype=dtype, device="cuda")
    buf[offset:offset + rows * ld].view(rows, ld)[:, :cols] = dev(m64, dtype)
    base = buf[offset:]
    am = np.abs(m64)
    ref, mag, k = (m64 @ m64.T, am @ am.T, cols) if side == 0 else (m64.T @ m64, am.T @ am, rows)
    simt = f"gemm_f64acc_kernel<{CNAME[dtype]}, {CNAME[dtype]}>"
    checks = [(0, route)] + ([(2, "simt")] if route == "dmma" else [])     # gram_path = 2: the same matrix on SIMT
    for path, want in checks:
        ctx.set_option("gram_path", path)
        with kernels() as ran:
            g = _gram(lib, base, rows, cols, ld, dtype, side)
        if want == "dmma":
            assert_ran(ran, ["gram_dmma_kernel", "gram_dmma_reduce_kernel"], ["gemm_f64acc_kernel", "gram_i8_kernel"])
        else:
            assert_ran(ran, simt, ["gram_dmma_kernel", "gram_i8_kernel"])
        got = g.cpu().numpy()
        assert_product(got, ref, mag, k, F64)
        assert np.array_equal(got, got.T), "not bitwise symmetric"


# ---- DCT -------------------------------------------------------------------------------------------------------
# ndmps_dct_last_axis is the product of the lines with the orthonormal cosine matrix: on gemm_tc_kernel (tcgen05) for
# float32 with lines * n >= 2^20 when gemm_tc takes the shape (n >= 8, lines >= 128), else through gemm(): DMMA when the
# tile rule allows, SIMT otherwise.
DCT_CASES = {f"{'f32' if dt == F32 else 'f64'}-37x{n}": (37, n, dt, "simt")     # id: (lines, n, dtype, route)
             for dt in (F32, F64) for n in (1, 2, 4, 25, 64, 65, 680)}
DCT_CASES.update({
    "f32-16383x64-dmma": (16383, 64, F32, "dmma128"),          # lines * n just under 2^20
    "f32-16384x64-tcgen05": (16384, 64, F32, "tc"),            # exactly 2^20
    "f32-262144x4-n-below-8": (262144, 4, F32, "simt"),              # large enough for tcgen05, too narrow for it
    "f64-20000x128-dmma": (20000, 128, F64, "dmma128"),
    "f64-16384x64-dmma": (16384, 64, F64, "dmma128"),          # float64 never takes tcgen05
})


def _dct_matrix(n):
    k, i = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    c = np.sqrt(2.0 / n) * np.cos(np.pi * (2 * i + 1) * k / (2 * n))
    c[0] *= np.sqrt(0.5)
    return c


@pytest.mark.parametrize("case", list(DCT_CASES), ids=str)
def test_dct_routes(lib, ctx, case):
    _, ops = lib
    lines, n, dtype, route = DCT_CASES[case]
    x64 = rounded(np.random.default_rng([lines, n]), (lines, n), dtype)
    ac = np.abs(_dct_matrix(n))
    if route == "tc":
        want, absent = ["gemm_tc_kernel"], ["gemm_dmma_kernel", "gemm_f64acc_kernel"]
    elif route == "dmma128":
        want = [f"gemm_dmma_kernel<128, {CNAME[dtype]}, double, {CNAME[dtype]}>"]
        absent = ["gemm_tc_kernel", "gemm_f64acc_kernel"]
    else:
        want, absent = [f"gemm_f64acc_kernel<{CNAME[dtype]}, double>"], ["gemm_tc_kernel", "gemm_dmma_kernel"]
    x = dev(x64, dtype)
    out = {}
    for inverse in (False, True):
        ref = (scipy_fft.idct if inverse else scipy_fft.dct)(x64, type=2, norm="ortho", axis=-1)
        mag = np.abs(x64) @ (ac if inverse else ac.T)
        with kernels() as ran:
            got = ops.dct_last_axis(x, inverse=inverse)
        assert_ran(ran, want, absent)
        if route == "tc":
            assert float(np.max(np.abs(got.double().cpu().numpy() - ref))) <= 1e-6 * np.max(np.abs(ref))
        else:
            # the device builds the cosine matrix with cospi: a few ulp per entry on top of the accumulation
            assert_product(got, ref, mag, n + 4, dtype)
        out[inverse] = got
    back = ops.dct_last_axis(out[False], inverse=True).double().cpu().numpy()
    tol = 1e-13 if dtype == F64 else 4e-6
    assert float(np.max(np.abs(back - x64))) <= tol * np.max(np.abs(x64))


# ---- reductions ------------------------------------------------------------------------------------------------
# reduce_stage1 (reduce.cu): float32 arrays whose pointers are 16-byte aligned take float4 loads, two in flight per
# thread, then single float4 loads, then a scalar tail of n % 4; float64 and misaligned float32 take the scalar
# grid-stride loop.  The grid has ceil(n / 2048) blocks of 256 threads, up to 8 per SM: past 2048 * 8 * sm_count
# elements every loop runs more than once per thread.
def _cap(sm):
    return 2048 * 8 * sm


RED_SIZES = {                    # id: n from the SM count
    "n1": lambda sm: 1, "n3": lambda sm: 3, "n4": lambda sm: 4, "n5": lambda sm: 5, "n1023": lambda sm: 1023,
    "n2048-one-block": lambda sm: 2048, "n2049-two-blocks": lambda sm: 2049,
    "grid-cap-1": lambda sm: _cap(sm) - 1, "grid-cap": _cap, "grid-cap+1": lambda sm: _cap(sm) + 1,
    "5x-grid-cap+7": lambda sm: 5 * _cap(sm) + 7,
}
RED_OFFSETS = {"aligned": (0, 0), "a+1-b+1": (1, 1), "a+2-b+2": (2, 2), "a+3-b+3": (3, 3), "b+1-only": (0, 1)}
RED_CASES = {f"{s}-{o}": (s, o) for s in RED_SIZES for o in RED_OFFSETS
             if o in ("aligned", "a+1-b+1", "b+1-only") or not s.startswith(("grid", "5x"))}


def placed(values, offset, dtype):
    """Device view of `values` starting `offset` elements into a fresh allocation padded with NaN on both sides."""
    buf = torch.full((offset + len(values) + 8,), float("nan"), dtype=dtype, device="cuda")
    assert buf.data_ptr() % 256 == 0
    view = buf[offset:offset + len(values)]
    if len(values):
        view.copy_(dev(values, dtype))
    return view


def fsum_sq(x):
    return math.fsum(np.square(x).tolist())


def _red_kernel(dtype, mode):
    return f"reduce_stage1<{CNAME[dtype]}, {mode}>"


@pytest.mark.parametrize("dtype", [F32, F64], ids=["f32", "f64"])
@pytest.mark.parametrize("case", list(RED_CASES), ids=str)
def test_reductions_sizes_and_offsets(lib, sm, case, dtype):
    _, ops = lib
    size, offsets = RED_CASES[case]
    n = RED_SIZES[size](sm)
    oa, ob = RED_OFFSETS[offsets]
    rng = np.random.default_rng([n, oa, ob])
    x64 = rounded(rng, n, dtype)
    y64 = (x64 + 0.01 * rng.standard_normal(n)).astype(NP[dtype]).astype(np.float64)
    a, b = placed(x64, oa, dtype), placed(y64, ob, dtype)
    with kernels() as ran:
        s = ops.sumsq(a)
    assert_ran(ran, _red_kernel(dtype, 0))
    assert abs(s - fsum_sq(x64)) <= 1e-13 * fsum_sq(x64)
    with kernels() as ran:
        mm = ops.minmax([a, b])
    assert_ran(ran, _red_kernel(dtype, 1))
    assert np.array_equal(mm, [[x64.min(), x64.max()], [y64.min(), y64.max()]])
    with kernels() as ran:
        sq, peak = ops.psnr_terms(a, b)
    assert_ran(ran, _red_kernel(dtype, 2))
    want = fsum_sq(x64 - y64)
    assert abs(sq - want) <= 1e-13 * want
    assert peak == x64.max()


def _fill(kind, n, rng):
    if kind == "extremes-in-scalar-tail":          # n % 4 == 3: the last three elements follow the float4 loads
        x = rng.standard_normal(n)
        x[-1], x[-2] = -50.0, 60.0
    elif kind == "extremes-in-last-float4":
        x = rng.standard_normal(n)
        x[-4], x[-5] = -50.0, 60.0
    elif kind == "all-negative":
        x = -0.5 - rng.random(n)
    elif kind == "constant":
        x = np.full(n, 0.375)
    else:                                          # float64 values float32 cannot represent (all round to 1.0f)
        x = 1.0 + 2.0 ** -30 * rng.random(n)
    return x


RED_FILLS = ["extremes-in-scalar-tail", "extremes-in-last-float4", "all-negative", "constant", "beyond-float32"]


@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("dtype", [F32, F64], ids=["f32", "f64"])
@pytest.mark.parametrize("size", ["n1027", "grid-cap+3"])
@pytest.mark.parametrize("fill", RED_FILLS)
def test_reductions_values(lib, sm, fill, size, dtype, offset):
    _, ops = lib
    n = 1027 if size == "n1027" else _cap(sm) + 3
    x64 = _fill(fill, n, np.random.default_rng(n)).astype(NP[dtype]).astype(np.float64)
    y64 = x64[::-1].copy()
    a, b = placed(x64, offset, dtype), placed(y64, offset, dtype)
    with kernels() as ran:
        s = ops.sumsq(a)
        mm = ops.minmax([a])
        sq, peak = ops.psnr_terms(a, b)
    assert_ran(ran, [_red_kernel(dtype, mode) for mode in (0, 1, 2)])
    assert abs(s - fsum_sq(x64)) <= 1e-13 * fsum_sq(x64)
    assert mm[0, 0] == x64.min() and mm[0, 1] == x64.max()
    want = fsum_sq(x64 - y64)
    assert abs(sq - want) <= 1e-13 * want
    assert peak == x64.max()


@pytest.mark.parametrize("dtype", [F32, F64], ids=["f32", "f64"])
def test_minmax_mixed_arrays_and_empty_sumsq(lib, sm, dtype):
    _, ops = lib
    rng = np.random.default_rng(5)
    sizes, offsets = [1, 5, 1023, 2049, _cap(sm) + 1, 4], [3, 0, 1, 2, 1, 0]
    # scaled before the rounding to `dtype`, so the float64 copies hold exactly what the device arrays hold
    xs = [(rng.standard_normal(n) * (i + 1)).astype(NP[dtype]).astype(np.float64) for i, n in enumerate(sizes)]
    with kernels() as ran:
        mm = ops.minmax([placed(x, o, dtype) for x, o in zip(xs, offsets)])
    assert_ran(ran, _red_kernel(dtype, 1))
    assert np.array_equal(mm, [[x.min(), x.max()] for x in xs])
    for empty in (placed(np.zeros(0), 1, dtype), torch.empty(0, dtype=dtype, device="cuda")):   # data_ptr() is 0
        with kernels() as ran:
            s = ops.sumsq(empty)
        assert_ran(ran, _red_kernel(dtype, 0))
        assert s == 0.0


# ---- quantisation ----------------------------------------------------------------------------------------------
INT_TYPES = {np.uint8: "unsigned char", np.uint16: "unsigned short", np.uint32: "unsigned int",
             np.uint64: "unsigned long", np.int8: "signed char", np.int16: "short", np.int32: "int", np.int64: "long"}
QUANT_SIZES = {"random-1000": 1000, "random-1e6+7": 10 ** 6 + 7, "constant-4099": 4099}


def quantise_ref(x64, dt):
    """``scale_to_dtype`` with the library's rule where numpy's cast is undefined: NaN (0 / 0, every element of a
    constant array) gives 0 for every type, and a value past the type's range (the top code 1.0 * max, which is 2^64
    or 2^63 in float64, for the 64-bit types) saturates to the type's maximum.  The kernel tests for NaN itself: the
    B200's conversion of NaN gives 0x80...0 for the 32- and 64-bit types.  numpy on x86-64 gives instead int32 NaN ->
    -2^31, uint64 NaN -> 2^63 and top code -> 0, int64 NaN and top code -> -2^63.  Everywhere else the result must be
    the oracle's, bit for bit."""
    info = np.iinfo(dt)
    with np.errstate(invalid="ignore", divide="ignore"):
        shifted = x64 - np.min(x64)
        v = shifted / np.max(shifted) * info.max           # the oracle's arithmetic
        oracle = OQ.scale_to_dtype(x64, dt)
    nan = np.isnan(v)
    over = v >= 2.0 ** (info.bits - (1 if info.min < 0 else 0))
    want = np.where(nan | over, 0.0, v).astype(dt)
    want[over] = info.max
    defined = ~(nan | over)
    assert np.array_equal(want[defined], oracle[defined])
    return want


@pytest.mark.parametrize("dtype", [F32, F64], ids=["f32", "f64"])
@pytest.mark.parametrize("size", list(QUANT_SIZES))
@pytest.mark.parametrize("dt", list(INT_TYPES), ids=lambda t: np.dtype(t).name)
def test_quantise_every_integer_type(lib, dt, size, dtype):
    _, ops = lib
    n = QUANT_SIZES[size]
    rng = np.random.default_rng(n)
    if size.startswith("constant"):
        x64 = np.full(n, 0.3).astype(NP[dtype]).astype(np.float64)
    else:
        x64 = (3.0 * rng.standard_normal(n) + 1.0).astype(NP[dtype]).astype(np.float64)
        x64[[7, n // 2]] = x64.min()                        # repeated extremes: exactly lo and exactly hi
        x64[[11, n - 1]] = x64.max()
    lo, hi = float(x64.min()), float(x64.max())
    code, qname = ops.int_code(dt), INT_TYPES[dt]
    want = quantise_ref(x64, dt)
    with kernels() as ran:
        q = ops.quantize(dev(x64, dtype), lo, hi, code)
    assert_ran(ran, f"quantize_kernel<{CNAME[dtype]}, {qname}>")
    got = ops.to_host_int(q, dt)
    assert got.dtype == np.dtype(dt)
    assert np.array_equal(got, want)
    if size.startswith("constant"):
        assert not got.any()
    back64 = OQ.scale_back(got, lo, hi, dt)
    for out in (F32, F64):
        with kernels() as ran:
            back = ops.dequantize(q, lo, hi, code, out)
        assert_ran(ran, f"dequantize_kernel<{CNAME[out]}, {qname}>")
        assert np.array_equal(back.cpu().numpy(), back64.astype(NP[out]))
