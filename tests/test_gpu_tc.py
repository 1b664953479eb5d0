"""The tcgen05 kernels (csrc/tc_gemm.cu) called directly through the C ABI, against float64 references on the same
seeded inputs.

* sliced-integer Gram (`gram_path = 3`): error-free int32 accumulation of five 7-bit digit planes: the result must be
  within 1e-10 (relative to the largest entry) of the float64 accumulation of the same float32 data, exactly symmetric,
  and heavy-tailed rows must be handed to the exact FP64-pipe kernel by the device-side flag (error 0);
* bf16x3 GEMM (`gemm_path = 3`): float32-class accuracy (1e-6 relative to the largest entry; measured 2e-7) for every
  operand-major combination, both output orders, ragged edges, persistent grids with more tiles than SMs;
* the capped float32 sweep with and without the tensor-core kernels (`tc`): same bonds, singular values within 1e-8 of
  sigma_1, reconstructions within 1e-5 (the parity bar of the path)."""
import ctypes as C
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


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


def _rand(shape, seed, dtype=torch.float32, shift=0.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.rand(shape, device="cuda", generator=g, dtype=torch.float64) - shift).to(dtype)


# ---- Gram ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,cols", [(512, 32768), (360, 8192), (64, 4096), (2560, 4096), (200, 2051 * 4)])
def test_gram_i8_matches_float64_accumulation(lib, ctx, rows, cols):
    _, ops = lib
    m = _rand((rows, cols), 100 + rows)
    want = m.double() @ m.double().T
    ctx.set_option("gram_path", 3)
    got = ops.gram(m)
    assert float((got - want).abs().max() / want.abs().max()) <= 1e-10
    assert float((got - got.T).abs().max()) == 0.0
    ctx.set_option("tc_waves", 2)                                    # another split-K partition: same bound
    got2 = ops.gram(m)
    assert float((got2 - want).abs().max() / want.abs().max()) <= 1e-10


def test_gram_i8_rows_over_six_decades(lib, ctx):
    _, ops = lib
    g = torch.Generator(device="cuda").manual_seed(7)
    m = (torch.randn((512, 16384), device="cuda", generator=g, dtype=torch.float32) *
         torch.logspace(0, -6, 512, device="cuda")[:, None].float())
    want = m.double() @ m.double().T
    ctx.set_option("gram_path", 3)
    got = ops.gram(m)
    # every row is scaled by its own power of two: small rows keep their relative accuracy
    rel_diag = ((got.diagonal() - want.diagonal()).abs() / want.diagonal()).max()
    assert float(rel_diag) <= 1e-9
    lam_w = torch.linalg.eigvalsh(want).flip(0)
    lam_g = torch.linalg.eigvalsh(got).flip(0)
    assert float(((lam_g[:64].clamp_min(0).sqrt() - lam_w[:64].clamp_min(0).sqrt()).abs() / lam_w[0].sqrt()).max()) <= 1e-9


def test_gram_i8_heavy_tailed_rows_take_the_exact_kernel(lib, ctx):
    """max / rms of a row beyond what five digits resolve (rho^2 > 4096): the device-side flag makes the digit kernels
    return at once and the FP64-pipe kernel, launched behind them, produce the result: identical to gram_path = 0."""
    _, ops = lib
    m = _rand((256, 16384), 9)
    m[:, 5] = 2000.0
    ctx.set_option("gram_path", 0)
    ctx.set_option("tc", 0)
    exact = ops.gram(m)
    ctx.set_option("tc", 1)
    ctx.set_option("gram_path", 3)
    got = ops.gram(m)
    assert torch.equal(got, exact)


# ---- GEMM ----------------------------------------------------------------------------------------------------
def _gemm(native, a, b, out_dtype, out_t):
    m, k = a.shape
    _, n = b.shape
    c = torch.empty((n, m) if out_t else (m, n), dtype=out_dtype, device="cuda")
    cx = native.context()
    cx.set_option("gemm_out_t", 1 if out_t else 0)
    try:
        native.check(native.load_library().ndmps_gemm(native.handle(), m, n, k, 1.0, native.ptr(a), native.dtype_code(a.dtype),
                                                      a.stride(0), a.stride(1), native.ptr(b), native.dtype_code(b.dtype),
                                                      b.stride(0), b.stride(1), native.ptr(c), native.dtype_code(out_dtype),
                                                      m if out_t else n), "ndmps_gemm")
    finally:
        cx.set_option("gemm_out_t", 0)
    return c.T if out_t else c


GEMM_CASES = [  # m, n, k, A stored MN-major, B stored MN-major, transposed output, dtype A, dtype B
    (32768, 64, 512, True, False, True, torch.float32, torch.float64),      # projection T = P^T M
    (4096, 45, 360, True, False, True, torch.float32, torch.float64),       # ragged n and k
    (4096, 4096, 64, False, True, False, torch.float32, torch.float32),     # final contraction: 1024 tiles on 148 CTAs
    (20000, 520, 64, False, True, False, torch.float32, torch.float32),     # ragged tiles on both edges, vector + scalar drain
    (1000, 200, 136, False, True, False, torch.float32, torch.float32),
    (640, 128, 320, False, False, False, torch.float32, torch.float32),     # both K-major
    (640, 72, 200, True, True, False, torch.float64, torch.float64),        # both MN-major, float64 in
    (16384, 128, 1024, True, False, True, torch.float32, torch.float64),    # chi = 128 projection
    (4099, 133, 64, False, True, False, torch.float32, torch.float32),      # ldc not a multiple of 4: scalar drain
]


@pytest.mark.parametrize("m,n,k,a_mn,b_mn,out_t,da,db", GEMM_CASES)
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.float64])
def test_gemm_tc_layouts(lib, ctx, m, n, k, a_mn, b_mn, out_t, da, db, out_dtype):
    native, _ = lib
    a = _rand((k, m) if a_mn else (m, k), 3 * m + n, da, shift=0.3)
    b = _rand((k, n) if b_mn else (n, k), 5 * m + k, db, shift=0.5)
    av = a.T if a_mn else a
    bv = b if b_mn else b.T
    want = av.double() @ bv.double()
    ctx.set_option("gemm_path", 3)
    got = _gemm(native, av, bv, out_dtype, out_t)
    assert float((got.double() - want).abs().max() / want.abs().max()) <= 1e-6


# ---- the sweep with and without the tensor-core kernels ---------------------------------------------------------
@pytest.mark.parametrize("shape,chi", [((128, 128, 128), 32), ((64, 96, 160), 64), ((256, 256, 64), 16)])
def test_capped_sweep_tc_on_off(lib, ctx, shape, chi):
    from imgcompressionmps.core.ndmps import NDMPS
    rng = np.random.default_rng(11)
    z, y, x = np.meshgrid(*[np.linspace(-1, 1, s) for s in shape], indexing="ij")
    vol = (np.exp(-3 * (x * x + 0.5 * y * y + 2 * z * z)) + 0.3 * np.sin(5 * x + 3 * y) * np.cos(4 * z)
           + 0.02 * rng.standard_normal(shape)).astype(np.float32)
    v = torch.from_numpy(vol).cuda()
    res = {}
    for tc in (0, 1):
        ctx.set_option("tc", tc)
        launches0 = ctx.stat("tc_launches")
        obj = NDMPS.from_tensor(v, max_bond=chi)
        rec = obj.to_tensor_device()
        res[tc] = (obj, rec, ctx.stat("tc_launches") - launches0)
    (o0, r0, l0), (o1, r1, l1) = res[0], res[1]
    assert l0 == 0 and l1 > 0                                        # the option really switches kernels
    assert o0.bond_sizes() == o1.bond_sizes()
    for s0, s1 in zip(o0.singular_values, o1.singular_values):
        assert np.max(np.abs(np.asarray(s0) - np.asarray(s1))) <= 1e-8 * np.asarray(s0)[0]
    assert float(torch.linalg.vector_norm((r1 - r0).double()) / torch.linalg.vector_norm(r0.double())) <= 1e-5


# ---- the sweep's digit hand-off ------------------------------------------------------------------------------------
def _sweep_kernels(ctx, v, **kw):
    """NDMPS.from_tensor(v, **kw), the names of the CUDA kernels a trace of it recorded, and how many tcgen05 kernels it
    launched (the library's own count: it holds even where the trace misses a record)."""
    from imgcompressionmps.core.ndmps import NDMPS
    launches0 = ctx.stat("tc_launches")
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        torch.cuda.synchronize()
        obj = NDMPS.from_tensor(v, **kw)
        torch.cuda.synchronize()
    return obj, [e.name for e in prof.events()], ctx.stat("tc_launches") - launches0


def test_capped_sweep_hands_the_gram_digits_to_its_projection(lib, ctx):
    # (32, 64, 4096) -> sites [32, 16, 16, 16, 64]: the first group's unfolding is 512 x 16384, eligible for the
    # sliced-integer Gram; every later unfolding has fewer than 2048 columns, so only the first step can use tcgen05:
    # its Gram on kind::i8 and its projection, two tcgen05 launches
    shape, chi = (32, 64, 4096), 16
    rng = np.random.default_rng(5)
    z, y, x = np.meshgrid(*[np.linspace(-1, 1, s) for s in shape], indexing="ij")
    vol = (np.exp(-3 * (x * x + 0.5 * y * y + 2 * z * z)) + 0.3 * np.sin(5 * x + 3 * y) * np.cos(4 * z)
           + 0.02 * rng.standard_normal(shape)).astype(np.float32)
    smooth = torch.from_numpy(vol).cuda()
    out_t = re.compile(r"gemm_tc_kernel<\d+, \d+, \w+, \w+, true, float>")    # bf16x3 product with transposed output

    # smooth rows: five digits are exact, the projection multiplies the digits the Gram made
    _, names, tc = _sweep_kernels(ctx, smooth, max_bond=chi)
    assert tc == 2
    for k in ("split_i8_proj_kernel", "proj_i8_kernel"):
        assert any(k in n for n in names), f"{k} did not run; kernels: {names}"
    assert not any(out_t.search(n) for n in names), names

    # one element 1e4 x the RMS: its row is too heavy-tailed for five digits, the device flag hands the Gram to the
    # FP64-pipe kernel and the projection to bf16x3 planes (the unfolding as the MN-major operand, T written transposed)
    spiky = smooth.clone()
    spiky[7, 33, 1000] = 1e4 * float(smooth.double().square().mean().sqrt())
    obj1, names, tc = _sweep_kernels(ctx, spiky, max_bond=chi)
    assert tc == 2
    assert not any("proj_i8_kernel" in n or "split_i8_proj_kernel" in n for n in names), names
    assert any(out_t.search(n) for n in names), names
    # the Gram the exact kernel computed is the one the sweep without tcgen05 computes: same first bonds
    ctx.set_option("tc", 0)
    obj0, _, tc = _sweep_kernels(ctx, spiky, max_bond=chi)
    ctx.set_option("tc", 1)
    assert tc == 0
    assert obj0.bond_sizes() == obj1.bond_sizes()
    s0, s1 = np.asarray(obj0.singular_values[0]), np.asarray(obj1.singular_values[0])
    assert np.max(np.abs(s0 - s1)) <= 1e-12 * s0[0]

    # an uncapped sweep and a float64 one keep to the FP64 pipe: no kernel of tc_gemm.cu (namespace ndmps::tc) runs
    for v, kw in ((smooth, {}), (smooth.double(), {"max_bond": chi})):
        _, names, tc = _sweep_kernels(ctx, v, **kw)
        assert tc == 0 and not any("ndmps::tc::" in n for n in names), names
