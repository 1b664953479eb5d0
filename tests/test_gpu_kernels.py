"""Kernel-level parity on a B200: every C-ABI building block against the oracle /
numpy on the same seeded inputs.  Bit-exact for integer / byte / index work
(permutation, quantisation), float tolerances stated per test."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from oracle import encoding as OE          # noqa: E402
from oracle import metrics as OM           # noqa: E402
from oracle import mps as OMPS             # noqa: E402
from oracle import quantise as OQ          # noqa: E402


@pytest.fixture(scope="module")
def ops():
    from imgcompressionmps import _ops
    return _ops


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


# ---- K1 permutation: bit exact --------------------------------------------------------------
SHAPES = [(8, 9), (4, 6), (7,), (1, 4), (12, 18, 10), (6, 10, 15), (4, 4, 4, 4), (16, 16, 8, 20), (30, 40, 50),
          (256, 128), (512, 680), (8, 512, 680), (64, 64, 64), (256, 256)]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_encode_decode_bit_exact(ops, shape, dtype):
    rng = np.random.default_rng(11)
    x = rng.standard_normal(shape).astype(dtype)
    want = OE.encode(x)
    got = ops.encode(dev(x))
    assert tuple(got.shape) == want.shape
    assert np.array_equal(got.cpu().numpy(), want)
    back = ops.decode(got, shape)
    assert np.array_equal(back.cpu().numpy(), x)


@pytest.mark.parametrize("shape", [(64, 64, 64), (256, 256), (256, 128), (32, 16, 8, 32), (128, 128, 128), (1024, 16)],
                         ids=lambda s: "x".join(map(str, s)))
def test_permutation_kernels_agree(ops, shape):
    """Power-of-two shapes: the register bit-permutation (default), the shared-memory tiles (permute_path = 1) and
    the gather kernel (2) give the oracle's permutation bit for bit, with and without the folded scale."""
    from imgcompressionmps import _native
    from imgcompressionmps.utils.core import get_factorlist
    factors, _ = get_factorlist(shape)
    assert _native.Plan(shape, factors).bit_info(False)["bits"]
    ctx = _native.context()
    x = np.random.default_rng(12).standard_normal(shape).astype(np.float32)
    want = OE.encode(x)
    try:
        for path in (0, 1, 2):
            ctx.set_option("permute_path", path)
            got = ops.encode(dev(x))
            assert np.array_equal(got.cpu().numpy(), want), path
            assert np.array_equal(ops.decode(got, shape).cpu().numpy(), x), path
            assert np.array_equal(ops.encode(dev(x), 0.375).cpu().numpy(), want * np.float32(0.375)), path
    finally:
        ctx.set_option("permute_path", 0)


def test_encode_golden_ramp(ops, golden_encoding):
    """Device permutation of a ramp == the reference's own scatter (fixtures made by running it)."""
    import hashlib
    g = golden_encoding
    for key in sorted({k.split("/")[0] for k in g.files}):
        shape = tuple(int(s) for s in key.split("x"))
        n = int(np.prod(shape))
        if f"{key}/encoded_ramp" in g.files:
            ramp = np.arange(n, dtype=np.float32).reshape(shape)
            got = ops.encode(dev(ramp)).cpu().numpy().astype(np.int32)
            assert np.array_equal(got, g[f"{key}/encoded_ramp"]), key
        elif f"{key}/encoded_ramp_sha256" in g.files and n < 2 ** 24:   # ramp exact in float32 below 2^24
            ramp = np.arange(n, dtype=np.float32).reshape(shape)
            got = ops.encode(dev(ramp)).cpu().numpy().astype(np.int32)
            assert hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest() == str(g[f"{key}/encoded_ramp_sha256"]), key


def test_encode_scale(ops):
    x = np.random.default_rng(0).random((12, 18, 10)).astype(np.float32)
    got = ops.encode(dev(x), 0.25).cpu().numpy()
    assert np.array_equal(got, OE.encode(x) * np.float32(0.25))


# ---- reductions ------------------------------------------------------------------------------
def test_reductions(ops):
    rng = np.random.default_rng(1)
    x = rng.standard_normal(1_000_003).astype(np.float32)
    y = (x + 0.01 * rng.standard_normal(x.size)).astype(np.float32)
    assert ops.sumsq(dev(x)) == pytest.approx(float(np.sum(x.astype(np.float64) ** 2)), rel=1e-13)
    mm = ops.minmax([dev(x), dev(y[:17])])
    assert np.array_equal(mm, [[x.min(), x.max()], [y[:17].min(), y[:17].max()]])
    sq, peak = ops.psnr_terms(dev(x), dev(y))
    assert sq == pytest.approx(float(np.sum((x.astype(np.float64) - y) ** 2)), rel=1e-12)
    assert peak == float(x.max())


# ---- GEMM / Gram -------------------------------------------------------------------------------
@pytest.mark.parametrize("m,n,k", [(1, 1, 1), (5, 7, 3), (64, 64, 16), (65, 130, 1000), (8, 8, 100_000), (512, 64, 300),
                                   (3, 1000, 5)])
def test_gemm_matches_numpy(ops, m, n, k):
    rng = np.random.default_rng(2)
    a = rng.standard_normal((m, k)).astype(np.float32)
    b = rng.standard_normal((k, n))
    want = a.astype(np.float64) @ b
    got = ops.gemm(dev(a), dev(b), out_dtype=torch.float64).cpu().numpy()
    assert np.allclose(got, want, rtol=1e-13, atol=1e-12 * np.abs(want).max())
    # transposed views go through the stride arguments, no copies
    got_t = ops.gemm(dev(b.T.copy()).t(), dev(a.T.copy()).t(), out_dtype=torch.float64).cpu().numpy() if False else None
    at = dev(np.ascontiguousarray(a.T)).t()       # logical (m, k), K-strided
    got2 = ops.gemm(at, dev(b), out_dtype=torch.float32).cpu().numpy()
    assert np.allclose(got2, want, rtol=2e-6, atol=2e-6 * np.abs(want).max())


@pytest.mark.parametrize("rows,cols", [(8, 4096), (64, 32768), (512, 2048), (100, 77), (20, 3000)])
def test_gram_float64_accumulation(ops, rows, cols):
    rng = np.random.default_rng(3)
    m = rng.standard_normal((rows, cols)).astype(np.float32)
    m64 = m.astype(np.float64)
    g0 = ops.gram(dev(m), 0).cpu().numpy()
    want0 = m64 @ m64.T
    assert np.allclose(g0, want0, rtol=0, atol=1e-13 * np.abs(want0).max())
    assert np.array_equal(g0, g0.T)                # bitwise symmetric by construction
    g1 = ops.gram(dev(m), 1).cpu().numpy()
    want1 = m64.T @ m64
    assert np.allclose(g1, want1, rtol=0, atol=1e-13 * np.abs(want1).max())


# ---- Jacobi eigensolver ---------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2, 3, 8, 33, 64, 100, 128, 129, 200, 512, 600])
def test_eigh_random_gram(ops, n):
    rng = np.random.default_rng(n)
    a = rng.standard_normal((n, 3 * n + 5))
    g = a @ a.T
    evals, evecs, sweeps = ops.eigh(dev(g))
    evals, evecs = evals.cpu().numpy(), evecs.cpu().numpy()
    want = np.linalg.eigvalsh(g)[::-1]
    assert np.all(np.diff(evals) <= 0)
    assert np.allclose(evals, want, rtol=0, atol=1e-12 * want[0])
    assert np.allclose(evecs.T @ evecs, np.eye(n), atol=1e-11)
    assert np.allclose(g @ evecs, evecs * evals[None, :], atol=1e-11 * want[0])
    print(f"eigh n={n}: {sweeps} sweeps")


@pytest.mark.parametrize("n", [64, 300, 512])
def test_eigh_graded_and_rank_deficient(ops, n):
    """Spectrum spanning 16 decades plus an exact null space: the sweep's rank decisions need
    eigenvalues resolved relative to lambda_max at the 1e-12 level."""
    rng = np.random.default_rng(100 + n)
    q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    lam = np.zeros(n)
    k = n // 2
    lam[:k] = 10.0 ** np.linspace(4, -12, k)
    g = (q * lam[None, :]) @ q.T
    g = 0.5 * (g + g.T)
    evals, evecs, sweeps = ops.eigh(dev(g))
    evals, evecs = evals.cpu().numpy(), evecs.cpu().numpy()
    assert np.allclose(evals[:k], lam[:k], rtol=0, atol=1e-12 * lam[0])
    big = lam[:k] > 1e-6 * lam[0]
    nb = int(big.sum())
    assert np.allclose(evals[:nb], lam[:nb], rtol=1e-8)
    # leading eigenvectors span the right subspace
    proj = q[:, :nb].T @ evecs[:, :nb]
    assert np.allclose(np.abs(np.diag(proj)), 1.0, atol=1e-6)
    print(f"graded n={n}: {sweeps} sweeps")


# ---- leading-eigenpair solver (capped bonds) -----------------------------------------------------
def _topk_check(ops, g, k, res_tol=1e-12):
    evals, evecs, trace, health = ops.eigh_topk(dev(g), k)
    evals, evecs = evals.cpu().numpy(), evecs.cpu().numpy()
    want = np.linalg.eigvalsh(g)[::-1]
    assert health == 0
    assert np.all(np.diff(evals) <= 0)
    assert np.allclose(evals, want[:k], rtol=0, atol=1e-13 * want[0])
    assert abs(trace - np.trace(g)) <= 1e-13 * np.trace(g)
    assert np.allclose(evecs.T @ evecs, np.eye(k), atol=1e-12)
    assert np.max(np.linalg.norm(g @ evecs - evecs * evals[None, :], axis=0)) <= res_tol * want[0]
    return evals, evecs


@pytest.mark.parametrize("n,k", [(96, 16), (200, 64), (256, 64), (357, 64), (512, 64), (512, 100), (512, 128), (1000, 64), (1024, 128), (1025, 64), (1536, 64), (2560, 64)])
def test_eigh_topk_random_gram(ops, n, k):
    rng = np.random.default_rng(7 * n + k)
    a = rng.standard_normal((n, 2 * n + 3))
    _topk_check(ops, a @ a.T, k)


@pytest.mark.parametrize("option,n", [("topk_cluster", 357), ("topk_cluster", 512)])
def test_eigh_topk_alternative_routes(ops, option, n):
    """The grid-barrier tridiagonalisation, which runs instead of the thread-block cluster when the cluster does not fit
    the device, stays correct for the sizes the cluster covers."""
    from imgcompressionmps import _native
    ctx = _native.context()
    rng = np.random.default_rng(3 * n + len(option))
    a = rng.standard_normal((n, 2 * n + 1)) * np.logspace(0, -3, n)[:, None]
    ctx.set_option(option, 0)
    try:
        _topk_check(ops, a @ a.T, 64)
    finally:
        ctx.set_option(option, 1)


@pytest.mark.parametrize("n", [256, 512])
def test_eigh_topk_clusters_and_rank_deficiency(ops, n):
    """Repeated and nearly repeated leading eigenvalues (the block is re-orthonormalised between
    inverse-iteration steps and rotated by Rayleigh-Ritz) and a null space behind the kept part."""
    rng = np.random.default_rng(n)
    q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    lam = np.zeros(n)
    lam[:16] = 5.0
    lam[16:32] = 5.0 - 1e-13
    lam[32:48] = 2.0 * (1.0 - 1e-9 * np.arange(16))
    lam[48:150] = 10.0 ** np.linspace(0, -9, 102)
    g = (q * lam[None, :]) @ q.T
    g = 0.5 * (g + g.T)
    evals, evecs = _topk_check(ops, g, 64, res_tol=5e-12)
    # the 48 leading vectors span the same subspace as the true ones
    proj = q[:, :48].T @ evecs[:, :48]
    assert np.allclose(np.linalg.svd(proj, compute_uv=False), 1.0, atol=1e-9)


def test_eigh_topk_rejects_unsupported_shapes(ops):
    g = np.eye(64)
    with pytest.raises(ValueError):
        ops.eigh_topk(dev(g), 8)          # n < 96
    with pytest.raises(ValueError):
        ops.eigh_topk(dev(np.eye(256)), 200)   # 2k > n


# ---- DCT --------------------------------------------------------------------------------------------
def test_dct_against_scipy_fftpack_fixture(ops, golden_dct):
    g = golden_dct
    for i in range(5):
        x = g[f"in{i}"]
        got = ops.dct_last_axis(dev(x)).cpu().numpy()
        assert np.allclose(got, g[f"dct{i}"], atol=1e-13), i
        got_i = ops.dct_last_axis(dev(x), inverse=True).cpu().numpy()
        assert np.allclose(got_i, g[f"idct{i}"], atol=1e-13), i
        x32 = x.astype(np.float32)
        got32 = ops.dct_last_axis(dev(x32)).cpu().numpy()
        assert np.allclose(got32, g[f"dct{i}"], atol=2e-6)


# ---- quantisation: bit exact --------------------------------------------------------------------------
def test_quantise_bit_exact(ops, golden_quantise):
    g = golden_quantise
    for i in range(3):
        a = g[f"in{i}"]
        for bits, dt in ((8, np.uint8), (16, np.uint16)):
            name = np.dtype(dt).name
            q = ops.quantize(dev(a), a.min(), a.max(), bits)
            assert np.array_equal(q.cpu().numpy(), g[f"q{i}_{name}"])
            back = ops.dequantize(q, a.min(), a.max(), bits, torch.float64).cpu().numpy()
            assert np.array_equal(back, g[f"back{i}_{name}"])
    # float32 cores: arithmetic in float64 on the exact float32 values, as the oracle would do after upcasting
    rng = np.random.default_rng(9)
    c = rng.standard_normal((40, 8, 33)).astype(np.float32)
    q = ops.quantize(dev(c), float(c.min()), float(c.max()), 16).cpu().numpy()
    assert np.array_equal(q, OQ.scale_to_dtype(c.astype(np.float64), np.uint16))


# ---- SSIM / PSNR ------------------------------------------------------------------------------------------
def _pair(shape, seed, dtype):
    rng = np.random.default_rng(seed)
    a = rng.random(shape)
    b = a + 0.08 * rng.standard_normal(shape) - 0.02        # some negatives -> exercises the clip
    return a.astype(dtype), b.astype(dtype)


import contextlib


@contextlib.contextmanager
def ssim_arithmetic(exact):
    """float32 inputs: float64 arithmetic (the reference's) when `exact`, else the default shifted / normalised float32."""
    from imgcompressionmps import _native
    ctx = _native.context()
    ctx.set_option("ssim_exact", 1 if exact else 0)
    try:
        yield
    finally:
        ctx.set_option("ssim_exact", 0)


# float64 arithmetic agrees with the oracle to rounding; the streaming kernels for float32 inputs (float64 window sums,
# float32 formula) to ~1e-7 (north-star bar: 1e-4)
SSIM_TOL = {True: 1e-10, False: 1e-6}


@pytest.mark.parametrize("shape", [(16, 16), (40, 70), (7, 9), (5, 30), (6, 31), (256, 256), (33, 65), (70, 100), (39, 38)])
@pytest.mark.parametrize("dtype,exact", [(np.float64, True), (np.float32, True), (np.float32, False)], ids=["f64", "f32-exact", "f32-fast"])
def test_ssim_2d(ops, shape, dtype, exact):
    a, b = _pair(shape, 1, dtype)
    want = OM.compute_ssim_2d(a.astype(np.float64), b.astype(np.float64))
    with ssim_arithmetic(exact):
        got = ops.ssim(dev(a), dev(b))
    assert got == pytest.approx(want, abs=SSIM_TOL[exact])


@pytest.mark.parametrize("shape", [(9, 10, 11), (32, 48, 40), (64, 64, 64), (37, 45, 50), (40, 71, 33)])
@pytest.mark.parametrize("exact", [True, False], ids=["exact", "fast"])
def test_ssim_3d(ops, shape, exact):
    a, b = _pair(shape, 2, np.float32)
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    with ssim_arithmetic(exact):
        assert ops.ssim(dev(a), dev(b)) == pytest.approx(OM.avg_ssim_3d(a64, b64), abs=SSIM_TOL[exact])
        for ax in range(3):
            got = ops.ssim_slices(dev(a), dev(b), ax)
            assert np.allclose(got, OM.ssim_3d_axis(a64, b64, ax), atol=SSIM_TOL[exact])


@pytest.mark.parametrize("shape", [(16, 12, 10, 5), (12, 10, 9, 40), (40, 39, 8, 33)])
@pytest.mark.parametrize("exact", [True, False], ids=["exact", "fast"])
def test_ssim_4d(ops, shape, exact):
    a, b = _pair(shape, 3, np.float32)
    want = OM.avg_ssim_4d(a.astype(np.float64), b.astype(np.float64))
    with ssim_arithmetic(exact):
        assert ops.ssim(dev(a), dev(b)) == pytest.approx(want, abs=SSIM_TOL[exact])


def test_ssim_fast_path_offsets_and_scales(ops):
    """The streaming kernels sum in float64 and evaluate the formula in float32 on range-normalised moments: large
    offsets, tiny and huge scales and a steep edge next to flat texture must stay within the documented 1e-6."""
    rng = np.random.default_rng(11)
    base = rng.random((96, 80))
    noisy = base + 0.03 * rng.standard_normal(base.shape)
    edge = base.copy()
    edge[:, 40:] += 5.0                                              # a step 5x the texture amplitude through every tile row
    for a64, b64 in ((base + 1000.0, noisy + 1000.0), (base * 1e-6, noisy * 1e-6), (base * 1e6, noisy * 1e6),
                     (edge, edge + 0.02 * rng.standard_normal(edge.shape))):
        a, b = a64.astype(np.float32), b64.astype(np.float32)
        want = OM.compute_ssim_2d(a.astype(np.float64), b.astype(np.float64))
        assert ops.ssim(dev(a), dev(b)) == pytest.approx(want, abs=1e-6)


# ---- contractions ------------------------------------------------------------------------------------------
def _random_mps(dims, ranks, seed, dtype=np.float64):
    rng = np.random.default_rng(seed)
    L = len(dims)
    cores = []
    for i in range(L):
        l = 1 if i == 0 else ranks[i - 1]
        r = 1 if i == L - 1 else ranks[i]
        shape = (dims[i], r) if i == 0 else ((l, dims[i]) if i == L - 1 else (l, dims[i], r))
        cores.append(rng.standard_normal(shape).astype(dtype))
    return cores


def test_contract_and_overlap(ops):
    dims, ra, rb = [6, 5, 4, 7, 3], [4, 9, 5, 2], [6, 3, 8, 3]
    a = _random_mps(dims, ra, 1)
    b = _random_mps(dims, rb, 2)
    da = ops.contract_dense([dev(c) for c in a]).cpu().numpy()
    assert np.allclose(da, OMPS.contract_dense(a), rtol=1e-12, atol=1e-12)
    got = ops.overlap([dev(c) for c in a], [dev(c) for c in b])
    assert got == pytest.approx(OMPS.overlap(a, b), rel=1e-12)
    a32 = [c.astype(np.float32) for c in a]
    got32 = ops.overlap([dev(c) for c in a32], [dev(c) for c in b])
    assert got32 == pytest.approx(OMPS.overlap([c.astype(np.float64) for c in a32], b), rel=1e-12)
    one = [np.arange(5.0)]
    assert ops.overlap([dev(one[0])], [dev(one[0])]) == pytest.approx(30.0)
    two = _random_mps([5, 6], [3], 4)
    assert np.allclose(ops.contract_dense([dev(c) for c in two]).cpu().numpy(), two[0] @ two[1])
