"""Bond truncation against the oracle: every quimb cutoff mode (abs, rel, sum2, rsum2, sum1, rsum1), renorm power
and bond cap of the sweep (ndmps_ttsvd, ndmps_roundtrip_host), the decision of the capped leading-eigenpair route,
and the pairwise truncation (ndmps_compress_bond, NDMPS.compress).

A rank comparison with the oracle only means something when no threshold sits within rounding of a compared
value.  So every case here is first run through the oracle's own rules step by step (``sweep_decisions``,
``compress_decisions``): the threshold must lie at least ``MIN_MARGIN`` (relative) away from every quantity the
rule compares it with, and where a bond cap binds, the kept values must lie at least as far above the first
dropped one (else the kept subspace is arbitrary).  The ``test_*_is_decidable`` tests check that on the host without a GPU; each GPU test
asserts it again before it compares.  The tie cases at the end are the exception: they pin the strict comparisons on
spectra the device reproduces exactly."""
import re
from functools import lru_cache

import numpy as np
import pytest

from conftest import phantom
from oracle import encoding as OE
from oracle import mps as M

MODES = ["abs", "rel", "sum2", "rsum2", "sum1", "rsum1"]
RENORM_DEFAULT = {"rsum2": 2, "sum2": 2, "rsum1": 1, "sum1": 1}
MIN_MARGIN = 1e-2
# float32 capped sweeps project on tcgen05 with errors of ~1e-8 s_0 (test_gpu_tc.py::test_capped_sweep_tc_on_off):
# the smallest kept singular value of every bond must be far above that
F32_CAPPED_MIN_KEPT = 1e-4
SV_TOL = {"f64": 1e-9, "f32": 1e-6}            # singular values, times s_0
REC_TOL = {"f64": 1e-8, "f32": 1e-5}           # reconstructions, relative
PRODUCT_TOL = {"f64": 1e-10, "f32": 1e-6}      # t1' t2' of compress_bond, relative
DTYPES = {"f64": np.float64, "f32": np.float32}


# ---------------------------------------------------------------------------------------------------------------
# decision margins from the oracle's rules
# ---------------------------------------------------------------------------------------------------------------
def decision_margin(s, cutoff, mode, max_bond=None):
    """Relative distance of the cutoff's threshold from the nearest quantity the rule compares with it: s itself
    for abs / rel, the reversed cumulative sums of s**p for the sum modes.  With a cap only the comparisons of the
    first max_bond values can change min(n_cut, max_bond).  A cutoff of 0 decides nothing (inf)."""
    if cutoff <= 0.0:
        return np.inf
    s = np.asarray(s, dtype=np.float64)
    if mode == "abs":
        q, thr = s, cutoff
    elif mode == "rel":
        q, thr = s, cutoff * s[0]
    else:
        sp = s ** (2 if mode.endswith("2") else 1)
        q, thr = np.cumsum(sp[::-1])[::-1], cutoff * (sp.sum() if mode.startswith("r") else 1.0)
    if max_bond:
        q = q[:max_bond]
    return float(np.min(np.abs(q - thr)) / thr)


def cap_gap(s, n, max_bond):
    """Where the cap binds, the kept subspace is only determined if s_n lies clearly below s_{n-1}: a cap through a
    (near-)degenerate pair picks an arbitrary mix of it, and the later bonds depend on that choice.  Relative gap
    1 - s_n / s_{n-1} there, inf elsewhere."""
    if not max_bond or n != max_bond or n >= len(s):
        return np.inf
    return float(1.0 - s[n] / s[n - 1])


def sweep_decisions(dense, dims, cutoff, mode, max_bond=None, renorm=None):
    """oracle.mps.tt_svd step by step (M._svd, M.n_keep, M.renorm_factor): per bond the full spectrum s, the kept
    count n, the decision margin and the gap at a binding cap."""
    if renorm is None:
        renorm = RENORM_DEFAULT.get(mode, 0)
    out = []
    r_prev = 1
    tm = np.asarray(dense, dtype=np.float64).reshape(dims[0], -1)
    for i in range(len(dims) - 1):
        _, s, vh = M._svd(tm.reshape(r_prev * dims[i], -1))
        n = M.n_keep(s, cutoff, mode, max_bond)
        f = M.renorm_factor(s, n, renorm)
        out.append({"s": s, "n": n, "margin": decision_margin(s, cutoff, mode, max_bond), "gap": cap_gap(s, n, max_bond)})
        tm = (s[:n] * f)[:, None] * vh[:n]
        r_prev = n
    return out


def compress_decisions(cores, cutoff, max_bond=None):
    """oracle.mps.compress_all bond by bond: the spectrum of the two-site matrix (that of R.L), kept count, margin."""
    cores = [np.array(c, dtype=np.float64) for c in cores]
    L = len(cores)
    out = []
    for i in range(1, L):
        a = cores[i - 1].reshape(-1, cores[i - 1].shape[-1])
        b = cores[i].reshape(cores[i].shape[0], -1)
        s = M._svd(a @ b)[1][:min(a.shape[0], a.shape[1], b.shape[1])]
        n = M.n_keep(s, cutoff, "rel", max_bond)
        out.append({"s": s, "n": n, "margin": decision_margin(s, cutoff, "rel", max_bond), "gap": cap_gap(s, n, max_bond)})
        cores[i - 1], cores[i], _ = M.compress_bond(cores[i - 1], cores[i], first=(i == 1), last=(i == L - 1),
                                                    cutoff=cutoff, max_bond=max_bond)
    return out


def assert_decidable(decisions, f32_capped=False):
    for i, d in enumerate(decisions):
        assert d["margin"] >= MIN_MARGIN, f"bond {i}: threshold within {d['margin']:.2e} of a compared value"
        assert d["gap"] >= MIN_MARGIN, f"bond {i}: the cap cuts between values {d['gap']:.2e} apart"
        if f32_capped:
            s = d["s"]
            assert s[d["n"] - 1] >= F32_CAPPED_MIN_KEPT * s[0], f"bond {i}: kept {s[d['n'] - 1] / s[0]:.1e} s_0"


# ---------------------------------------------------------------------------------------------------------------
# inputs and oracle results (cached: the host check and the GPU tests share them)
# ---------------------------------------------------------------------------------------------------------------
@lru_cache(maxsize=None)
def volume(shape, dt, seed=2026):
    """The phantom in the payload dtype, as float64 (what the oracle sees)."""
    return phantom(shape, seed=seed, background=0.01).astype(DTYPES[dt]).astype(np.float64)


@lru_cache(maxsize=None)
def dense_of(shape, dt):
    return OE.encode(volume(shape, dt))


@lru_cache(maxsize=None)
def decisions_of(shape, dt, cutoff, mode, max_bond, renorm):
    d = dense_of(shape, dt)
    return sweep_decisions(d, list(d.shape), cutoff, mode, max_bond, renorm)


@lru_cache(maxsize=None)
def oracle_sweep(shape, dt, cutoff, mode, max_bond, renorm):
    d = dense_of(shape, dt)
    return M.tt_svd(d, list(d.shape), cutoff=cutoff, cutoff_mode=mode, max_bond=max_bond, renorm=renorm,
                    return_svals=True)


def bond_inputs(t1_shape, t2_shape, sigma, seed, dt):
    """Cores whose two-site matrix has the singular values sigma: t1 = U diag(sigma) W R, t2 = R^-1 W^T V^T with
    U, V, W^T isometries and R an invertible gauge (condition number 4) from seeded QR factors.  Rounded to dt."""
    rng = np.random.default_rng(seed)
    a, r, b = int(np.prod(t1_shape[:-1])), t1_shape[-1], int(np.prod(t2_shape[1:]))
    k = len(sigma)
    assert k == min(a, r, b)
    U = np.linalg.qr(rng.standard_normal((a, k)))[0]
    V = np.linalg.qr(rng.standard_normal((b, k)))[0]
    W = np.linalg.qr(rng.standard_normal((r, k)))[0].T
    R = np.linalg.qr(rng.standard_normal((r, r)))[0] * np.linspace(0.5, 2.0, r)[None, :]
    t1 = (U * sigma) @ W @ R
    t2 = np.linalg.solve(R, W.T @ V.T)
    rnd = lambda t, shp: t.astype(DTYPES[dt]).astype(np.float64).reshape(shp)
    return rnd(t1, t1_shape), rnd(t2, t2_shape)


def cutoff_keeping(sigma, mode, n):
    """The cutoff of `mode` whose threshold lies half way (geometric for abs / rel) between the comparisons that
    keep n and n + 1 values of the descending spectrum sigma."""
    sigma = np.asarray(sigma, dtype=np.float64)
    if mode in ("abs", "rel"):
        thr = np.sqrt(sigma[n - 1] * sigma[n])
        return thr if mode == "abs" else thr / sigma[0]
    sp = sigma ** (2 if mode.endswith("2") else 1)
    tail = np.cumsum(sp[::-1])[::-1]                       # tail[i] = sum_{j >= i} sp[j]
    target = 0.5 * (tail[n - 1] + tail[n])
    return target / sp.sum() if mode.startswith("r") else target


# ---------------------------------------------------------------------------------------------------------------
# case tables
# ---------------------------------------------------------------------------------------------------------------
# (64,64,64): site dims [8]*6, the first three sites merge into one group of D = 512 (a decision at sub-step j
# changes P of sub-step j + 1).  (30,40,50): dims [20,60,50], the second step takes the column-side Gram (D > C).
# (8,9): dims [6,12], the two-site case.
SWEEP_CUTOFFS = {
    (64, 64, 64): {"abs": 1.0, "rel": 1e-2, "sum2": 1e-2, "rsum2": 2e-3, "sum1": 5e-2, "rsum1": 1e-4},
    (30, 40, 50): {"abs": 1.0, "rel": 1e-2, "sum2": 0.3, "rsum2": 1e-4, "sum1": 0.5, "rsum1": 1e-2},
    (8, 9): {"abs": 1.0, "rel": 0.2, "sum2": 0.1, "rsum2": 1e-2, "sum1": 1.0, "rsum1": 0.1},
}
SWEEP_RULES = [(m, None) for m in MODES] + [("rsum2", 0), ("rsum2", 1)]
SWEEP_CASES = [(shape, mode, renorm, dt) for shape in SWEEP_CUTOFFS for mode, renorm in SWEEP_RULES for dt in DTYPES]


def _sweep_id(c):
    shape, mode, renorm, dt = c
    return f"{'x'.join(map(str, shape))}-{mode}-renorm{'default' if renorm is None else renorm}-{dt}"


def _renorm(mode, renorm):
    return RENORM_DEFAULT.get(mode, 0) if renorm is None else renorm


# Capped route (capped_eigh in csrc/ttsvd.cu).  On 64^3 at chi = 16 it runs once, at the third sub-step of the merged
# group (an 8 * 16 = 128 row Gram); on (32,32,16,200) at chi = 32 once, on the 1024 x 1024 column-side Gram.
# name -> (shape, chi, mode, cutoff, renorm, route the verbose line must report)
REGIMES = {
    "a-rsum2-cap-binds": ((64, 64, 64), 16, "rsum2", 1e-10, None, "cap binds"),
    "a-sum2-absolute-cap-binds": ((64, 64, 64), 16, "sum2", 1e-2, None, "cap binds"),
    "b-cutoff-below-cap": ((64, 64, 64), 16, "rsum2", 5e-3, None, "full solver"),
    "c-tail-within-twice-target": ((64, 64, 64), 16, "rsum2", "tail/1.5", None, "full solver"),
    "d-rsum2-renorm0": ((64, 64, 64), 16, "rsum2", 1e-10, 0, "cap binds"),
    "column-side-rsum2": ((32, 32, 16, 200), 32, "rsum2", 1e-10, None, "cap binds"),
}
CAPPED_BOND = {(64, 64, 64): 2, (32, 32, 16, 200): 1}


@lru_cache(maxsize=None)
def regime_case(name):
    """(shape, chi, mode, cutoff, renorm, route) with regime (c)'s cutoff derived from the float64 oracle spectrum
    at the capped bond: target = tail_k / 1.5 puts the discarded weight in (target, 2 target]."""
    shape, chi, mode, cutoff, renorm, route = REGIMES[name]
    if cutoff == "tail/1.5":
        lam = decisions_of(shape, "f64", 1e-10, mode, chi, renorm)[CAPPED_BOND[shape]]["s"] ** 2
        cutoff = float(lam[chi:].sum() / 1.5 / lam.sum())
    return shape, chi, mode, cutoff, renorm, route


# compress_bond: (t1 core shape, t2 core shape) -> first / last core matricisations by their rank
BOND_SHAPES = {
    "first-last": ((24, 16), (16, 20)),
    "a<r": ((6, 10), (10, 4, 5)),                  # G1 = t1^T t1 is rank-deficient (6 of 10)
    "r>b": ((3, 4, 12), (12, 8)),                  # G2 = t2 t2^T is rank-deficient (8 of 12)
    "r=1": ((2, 3, 1), (1, 4, 2)),
    "middle-middle": ((4, 5, 12), (12, 6, 5)),
}
# (shape name, mode, renorm, max_bond): all modes and renorm powers on one shape, the cap binding and not binding,
# then every shape with three rules
BOND_RULES = ([("first-last", m, p, None) for m in MODES for p in (0, 1, 2)]
              + [("first-last", "rsum2", 2, 4), ("first-last", "abs", 0, 12), ("first-last", "sum1", 1, 3)]
              + [(s, m, p, None) for s in BOND_SHAPES if s != "first-last" for m, p in (("rel", 0), ("sum2", 2), ("rsum1", 1))])
BOND_CASES = [rule + (dt,) for rule in BOND_RULES for dt in DTYPES]


def _bond_id(c):
    shape, mode, renorm, max_bond, dt = c
    return f"{shape}-{mode}-renorm{renorm}-chi{max_bond or 0}-{dt}"


@lru_cache(maxsize=None)
def bond_case(shape_name, mode, max_bond, dt):
    """Inputs with the spectrum 0.6**i and the cutoff keeping about half of it (for r = 1 a cutoff far above the
    only value: at least one is always kept)."""
    t1_shape, t2_shape = BOND_SHAPES[shape_name]
    k = min(int(np.prod(t1_shape[:-1])), t1_shape[-1], int(np.prod(t2_shape[1:])))
    sigma = 0.6 ** np.arange(k)
    cutoff = cutoff_keeping(sigma, mode, max(k // 2, 1)) if k > 1 else {"abs": 10.0, "rel": 10.0}.get(mode, 10.0)
    t1, t2 = bond_inputs(t1_shape, t2_shape, sigma, seed=k, dt=dt)
    a = t1.reshape(-1, t1.shape[-1])
    b = t2.reshape(t2.shape[0], -1)
    s = M._svd(a @ b)[1][:k]
    return t1, t2, cutoff, s


# NDMPS.compress(cutoff, max_bond=chi) on a lossless float64 MPS of the 32^3 phantom (site dims [8]*5)
COMPRESS_CUTOFF = 1e-2
COMPRESS_CHIS = {"binds": 8, "does-not-bind": 64}


@lru_cache(maxsize=None)
def compress_oracle(chi):
    from oracle.ndmps import OracleNDMPS
    o = OracleNDMPS.from_tensor(volume((32, 32, 32), "f64"))
    decisions = compress_decisions(o.cores, COMPRESS_CUTOFF, chi)
    o.compress(COMPRESS_CUTOFF, max_bond=chi)
    return o, decisions


# the input test_gpu_sharded.py::test_sharded_world1_equals_plain_sweep adds with a cutoff binding below chi
SHARDED_CUTOFF_CASE = ((64, 64, 64), 16, 4e-3)


# ---------------------------------------------------------------------------------------------------------------
# 1. every case is decidable (host only)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", SWEEP_CASES, ids=_sweep_id)
def test_sweep_case_is_decidable(case):
    shape, mode, renorm, dt = case
    decisions = decisions_of(shape, dt, SWEEP_CUTOFFS[shape][mode], mode, None, renorm)
    assert_decidable(decisions)
    uncut = decisions_of(shape, dt, 0.0, mode, None, None)
    assert [d["n"] for d in decisions] != [d["n"] for d in uncut], "the cutoff truncates nothing"


@pytest.mark.parametrize("name", list(REGIMES))
@pytest.mark.parametrize("dt", list(DTYPES))
def test_capped_regime_is_decidable(name, dt):
    """Besides the margins: the capped bond's Gram is large enough for the route (mj >= 96, mj >= 4 chi), and the
    oracle spectrum there puts the case in the regime its name says."""
    shape, chi, mode, cutoff, renorm, route = regime_case(name)
    decisions = decisions_of(shape, dt, cutoff, mode, chi, renorm)
    assert_decidable(decisions, f32_capped=dt == "f32")
    j = CAPPED_BOND[shape]
    dims = list(dense_of(shape, dt).shape)
    rows = (decisions[j - 1]["n"] if j else 1) * dims[j]
    mj = min(rows, int(np.prod(dims[j + 1:])))                # the Gram is taken on the shorter side
    assert mj >= 96 and mj >= 4 * chi
    lam = decisions[j]["s"] ** 2
    tail = lam[chi:].sum()
    target = cutoff * (lam.sum() if mode == "rsum2" else 1.0)
    n = decisions[j]["n"]
    if name.startswith("b-"):
        assert n < chi
    elif name.startswith("c-"):
        assert n == chi and 1.2 * target < tail < 1.8 * target
    else:
        assert n == chi and tail > 4 * target


@pytest.mark.parametrize("case", BOND_CASES, ids=_bond_id)
def test_bond_case_is_decidable(case):
    shape, mode, renorm, max_bond, dt = case
    _, _, cutoff, s = bond_case(shape, mode, max_bond, dt)
    assert decision_margin(s, cutoff, mode, max_bond) >= MIN_MARGIN


@pytest.mark.parametrize("chi", list(COMPRESS_CHIS.values()), ids=list(COMPRESS_CHIS))
def test_compress_case_is_decidable(chi):
    assert_decidable(decisions_of((32, 32, 32), "f64", 1e-10, "rsum2", None, None))     # the MPS it starts from
    o, decisions = compress_oracle(chi)
    assert_decidable(decisions)
    binds = any(d["n"] == chi < M.n_keep(d["s"], COMPRESS_CUTOFF, "rel") for d in decisions)
    assert binds == (chi == COMPRESS_CHIS["binds"])


def test_sharded_cutoff_case_is_decidable():
    shape, chi, cutoff = SHARDED_CUTOFF_CASE
    x = phantom(shape, seed=3, background=0.01).astype(np.float32).astype(np.float64)
    d = OE.encode(x)
    decisions = sweep_decisions(d, list(d.shape), cutoff, "rsum2", chi)
    assert_decidable(decisions, f32_capped=True)
    uncut = sweep_decisions(d, list(d.shape), 1e-10, "rsum2", chi)
    assert any(a["n"] < b["n"] for a, b in zip(decisions, uncut)), "the cutoff must bind below chi somewhere"


# ---------------------------------------------------------------------------------------------------------------
# 2. the sweep: every mode and renorm, merged groups, column-side steps, two sites
# ---------------------------------------------------------------------------------------------------------------
def _torch():
    return pytest.importorskip("torch")


def _check_sweep(got_cores, ranks, svals, want, dt):
    from imgcompressionmps import _ops
    want_cores, want_svals = want
    assert ranks == M.bond_sizes(want_cores)
    for i, (sg, so) in enumerate(zip(svals, want_svals)):
        assert sg.shape == so.shape
        assert np.max(np.abs(sg - so)) <= SV_TOL[dt] * so[0], f"bond {i}"
    rec = _ops.contract_dense(got_cores).double().cpu().numpy()
    ro = M.contract_dense(want_cores)
    assert np.linalg.norm(rec - ro) / np.linalg.norm(ro) < REC_TOL[dt]


@pytest.mark.gpu
@pytest.mark.parametrize("case", SWEEP_CASES, ids=_sweep_id)
def test_sweep_matches_oracle(case):
    from imgcompressionmps import _ops
    torch = _torch()
    shape, mode, renorm, dt = case
    cutoff = SWEEP_CUTOFFS[shape][mode]
    assert_decidable(decisions_of(shape, dt, cutoff, mode, None, renorm))
    d = dense_of(shape, dt)
    dense = torch.from_numpy(d.astype(DTYPES[dt])).cuda()
    cores, ranks, svals = _ops.ttsvd(dense, list(d.shape), cutoff=cutoff, cutoff_mode=mode, renorm=renorm)
    assert cores[0].dtype == dense.dtype
    _check_sweep(cores, ranks, svals, oracle_sweep(shape, dt, cutoff, mode, None, _renorm(mode, renorm)), dt)


@pytest.mark.gpu
@pytest.mark.parametrize("case", SWEEP_CASES, ids=_sweep_id)
def test_roundtrip_host_matches_oracle(case):
    from imgcompressionmps import _ops
    shape, mode, renorm, dt = case
    cutoff = SWEEP_CUTOFFS[shape][mode]
    assert_decidable(decisions_of(shape, dt, cutoff, mode, None, renorm))
    x = volume(shape, dt).astype(DTYPES[dt])
    extras = {}
    rec, ranks = _ops.roundtrip_host(x, cutoff=cutoff, cutoff_mode=mode, renorm=renorm, extras=extras)
    want_cores, _ = oracle_sweep(shape, dt, cutoff, mode, None, _renorm(mode, renorm))
    assert ranks == M.bond_sizes(want_cores)
    assert extras["norm"] == pytest.approx(np.sqrt(M.overlap(want_cores, want_cores)), rel=REC_TOL[dt])
    ro = OE.decode(M.contract_dense(want_cores), shape)
    assert np.linalg.norm(rec.astype(np.float64) - ro) / np.linalg.norm(ro) < REC_TOL[dt]


# ---------------------------------------------------------------------------------------------------------------
# 3. the capped route's decision
# ---------------------------------------------------------------------------------------------------------------
CAPPED_LINE = re.compile(r"\[ndmps\] capped eigh n = (\d+), k = (\d+):.*-> (cap binds|full solver)")


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(REGIMES))
@pytest.mark.parametrize("dt", list(DTYPES))
def test_capped_route_regime(name, dt, capfd):
    """The leading-eigenpair route is taken only where the cap provably binds; wherever it declines the full solver
    must reproduce the cutoff's ranks.  Either way eig_topk 1 and 0 give the same ranks and singular values, and both
    match the oracle."""
    from imgcompressionmps import _native, _ops
    torch = _torch()
    shape, chi, mode, cutoff, renorm, route = regime_case(name)
    decisions = decisions_of(shape, dt, cutoff, mode, chi, renorm)
    assert_decidable(decisions, f32_capped=dt == "f32")
    d = dense_of(shape, dt)
    dense = torch.from_numpy(d.astype(DTYPES[dt])).cuda()
    ctx = _native.context()
    runs = {}
    try:
        ctx.set_option("verbose", 1)
        for topk in (1, 0):
            ctx.set_option("eig_topk", topk)
            capfd.readouterr()
            cores, ranks, svals = _ops.ttsvd(dense, list(d.shape), cutoff=cutoff, cutoff_mode=mode, max_bond=chi,
                                             renorm=renorm)
            runs[topk] = (cores, ranks, svals, capfd.readouterr().err)
    finally:
        ctx.set_option("eig_topk", 1)
        ctx.set_option("verbose", 0)
    j = CAPPED_BOND[shape]
    mj = min((decisions[j - 1]["n"] if j else 1) * d.shape[j], int(np.prod(d.shape[j + 1:])))
    print(name, dt, [ln for ln in runs[1][3].splitlines() if "capped eigh" in ln])
    assert CAPPED_LINE.findall(runs[1][3]) == [(str(mj), str(chi), route)]
    assert "capped eigh" not in runs[0][3]
    (c1, r1, s1, _), (c0, r0, s0, _) = runs[1], runs[0]
    assert r1 == r0 == [x["n"] for x in decisions]
    for a, b in zip(s1, s0):
        assert np.max(np.abs(a - b)) <= SV_TOL[dt] * b[0]
    want = oracle_sweep(shape, dt, cutoff, mode, chi, _renorm(mode, renorm))
    _check_sweep(c1, r1, s1, want, dt)
    _check_sweep(c0, r0, s0, want, dt)


# ---------------------------------------------------------------------------------------------------------------
# 4. compress_bond and NDMPS.compress(max_bond=...)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", BOND_CASES, ids=_bond_id)
def test_compress_bond_matches_oracle(case):
    """Rank exact, kept singular values and the product t1' t2' as the oracle's, and the weight split evenly
    (absorb="both"): t1'^T t1' = t2' t2'^T = diag(s_kept)."""
    from imgcompressionmps import _ops
    torch = _torch()
    shape, mode, renorm, max_bond, dt = case
    t1, t2, cutoff, s = bond_case(shape, mode, max_bond, dt)
    assert decision_margin(s, cutoff, mode, max_bond) >= MIN_MARGIN
    first, last = t1.ndim == 2, t2.ndim == 2
    w1, w2, ws = M.compress_bond(t1, t2, first, last, cutoff, cutoff_mode=mode, max_bond=max_bond, renorm=renorm)
    dev = lambda t: torch.from_numpy(np.ascontiguousarray(t).astype(DTYPES[dt])).cuda()
    g1, g2, gs = _ops.compress_bond(dev(t1.reshape(-1, t1.shape[-1])), dev(t2.reshape(t2.shape[0], -1)), cutoff,
                                    mode, max_bond, renorm)
    n = len(ws)
    assert g1.shape[1] == g2.shape[0] == len(gs) == n
    tol = SV_TOL[dt] * ws[0]
    assert np.max(np.abs(gs - ws)) <= tol
    a, b = g1.double().cpu().numpy(), g2.double().cpu().numpy()
    want = w1.reshape(-1, n) @ w2.reshape(n, -1)
    assert np.linalg.norm(a @ b - want) / np.linalg.norm(want) < PRODUCT_TOL[dt]
    assert np.max(np.abs(a.T @ a - np.diag(ws))) <= tol
    assert np.max(np.abs(b @ b.T - np.diag(ws))) <= tol


@pytest.mark.gpu
def test_compress_bond_resolution_limit():
    """ndmps.h: kept singular values below 1e-8 s_0 are below the resolution of the Gram route and come out as zero
    columns of t1' / rows of t2'; the product stays within about 1e-8 s_0 of the exact one.  (Which of those tiny
    values count as kept is not resolved either, so the rank is not compared with the oracle's.)"""
    from imgcompressionmps import _ops
    torch = _torch()
    sigma = np.array([1.0, 1e-1, 1e-2, 1e-3, 1e-4, 1e-5, 1e-6, 1e-7, 5e-9, 1e-10, 1e-11, 1e-12])
    t1, t2 = bond_inputs((30, 12), (12, 25), sigma, seed=5, dt="f64")
    g1, g2, gs = _ops.compress_bond(torch.from_numpy(t1).cuda(), torch.from_numpy(t2).cuda(), 1e-12, "rel")
    a, b = g1.cpu().numpy(), g2.cpu().numpy()
    assert len(gs) >= 7 and np.max(np.abs(gs[:7] - sigma[:7])) <= SV_TOL["f64"] * sigma[0]
    tiny = gs <= 1e-8 * gs[0]
    assert np.all(a[:, tiny] == 0.0) and np.all(b[tiny, :] == 0.0)
    assert np.linalg.norm(a @ b - t1 @ t2) <= 3e-8 * sigma[0]


@pytest.mark.gpu
@pytest.mark.parametrize("chi", list(COMPRESS_CHIS.values()), ids=list(COMPRESS_CHIS))
def test_ndmps_compress_max_bond_matches_oracle(chi):
    from imgcompressionmps.core.ndmps import NDMPS
    o, decisions = compress_oracle(chi)
    assert_decidable(decisions)
    g = NDMPS.from_tensor(volume((32, 32, 32), "f64"))
    g.compress(COMPRESS_CUTOFF, max_bond=chi)
    assert g.bond_sizes() == o.bond_sizes() == [d["n"] for d in decisions]
    for sg, so in zip(g.singular_values, o.last_svals):
        assert np.max(np.abs(sg - so)) <= SV_TOL["f64"] * so[0]
    ro = o.to_tensor()
    assert np.linalg.norm(g.to_tensor() - ro) / np.linalg.norm(ro) < REC_TOL["f64"]
    assert g.norm_value == pytest.approx(o.norm_value, rel=1e-9)


# ---------------------------------------------------------------------------------------------------------------
# 5. ties and rejected arguments
# ---------------------------------------------------------------------------------------------------------------
TIE_SPECTRUM = np.array([8.0, 4.0, 2.0, 1.0, 0.5])
# each threshold equals a compared quantity exactly: s = 1 (abs), 0.125 * 8 = 1 (rel), 0.25 + 1 (sum2),
# 0.5 + 1 (sum1).  quimb keeps s > cutoff strictly and stops the sums at the first value pushing them strictly above
# the target, so all four keep 3.
TIES = [("abs", 1.0), ("rel", 0.125), ("sum2", 1.25), ("sum1", 1.5)]


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(DTYPES))
def test_ties_sweep(dt):
    """The Jacobi solver does no rotation on a diagonal Gram, so the device spectrum is exact and the strict
    comparisons are decided on exactly the tied values."""
    from imgcompressionmps import _ops
    torch = _torch()
    dense = torch.from_numpy(np.diag(TIE_SPECTRUM).astype(DTYPES[dt])).cuda()
    _, ranks, svals = _ops.ttsvd(dense, [5, 5], cutoff=0.0, cutoff_mode="rel")
    assert ranks == [5] and np.array_equal(svals[0], TIE_SPECTRUM)
    for mode, cutoff in TIES:
        assert M.n_keep(TIE_SPECTRUM, cutoff, mode) == 3
        cores, ranks, svals = _ops.ttsvd(dense, [5, 5], cutoff=cutoff, cutoff_mode=mode)
        want_cores, want_svals = M.tt_svd(np.diag(TIE_SPECTRUM), [5, 5], cutoff=cutoff, cutoff_mode=mode,
                                          return_svals=True)
        assert ranks == [3], mode
        assert np.allclose(svals[0], want_svals[0], rtol=1e-15, atol=0), mode
        rec = _ops.contract_dense(cores).double().cpu().numpy()
        assert np.allclose(rec, M.contract_dense(want_cores), rtol=0, atol=SV_TOL[dt] * 8), mode


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(DTYPES))
def test_ties_compress_bond(dt):
    from imgcompressionmps import _ops
    torch = _torch()
    t1 = torch.eye(5, dtype=torch.float64 if dt == "f64" else torch.float32).cuda()
    t2 = torch.from_numpy(np.diag(TIE_SPECTRUM).astype(DTYPES[dt])).cuda()
    _, _, s = _ops.compress_bond(t1, t2, 0.0, "rel")
    assert np.array_equal(s, TIE_SPECTRUM)
    for mode, cutoff in TIES:
        g1, g2, s = _ops.compress_bond(t1, t2, cutoff, mode)
        assert len(s) == 3 and np.array_equal(s, TIE_SPECTRUM[:3]), mode
        product = g1.double().cpu().numpy() @ g2.double().cpu().numpy()
        assert np.allclose(product, np.diag(np.r_[TIE_SPECTRUM[:3], 0.0, 0.0]), rtol=0, atol=SV_TOL[dt] * 8), mode


@pytest.mark.gpu
@pytest.mark.parametrize("bad_mode", [0, 7])
def test_cutoff_mode_out_of_range_is_rejected(bad_mode):
    import ctypes as C
    from imgcompressionmps import _native as N
    from imgcompressionmps import _ops
    torch = _torch()
    lib = N.load_library()
    x = np.random.default_rng(0).random((8, 9))
    dense = torch.from_numpy(x.reshape(6, 12)).cuda()
    bufs = [torch.empty(72, dtype=torch.float64, device="cuda") for _ in range(2)]
    ranks = (C.c_int64 * 1)()
    rc = lib.ndmps_ttsvd(N.handle(), N.ptr(dense), N.F64, 2, N.i64_array([6, 12]), 1e-10, bad_mode, 0, 0,
                         N.ptr_array(bufs), N.i64_array([72, 72]), ranks, None, 0)
    with pytest.raises(ValueError, match="cutoff_mode"):
        N.check(rc, "ndmps_ttsvd")
    t1, t2 = dense[:, :6].contiguous(), dense[:, 6:].contiguous()
    n = C.c_int64(0)
    rc = lib.ndmps_compress_bond(N.handle(), N.ptr(t1), N.ptr(t2), N.F64, 6, 6, 6, 0.1, bad_mode, 0, 0,
                                 N.ptr(bufs[0]), N.ptr(bufs[1]), C.byref(n), None)
    with pytest.raises(ValueError, match="cutoff_mode"):
        N.check(rc, "ndmps_compress_bond")
    out = np.empty_like(x)
    rc = lib.ndmps_roundtrip_host(N.handle(), _ops.plan_for(x.shape).handle, x.ctypes.data_as(C.c_void_p),
                                  out.ctypes.data_as(C.c_void_p), N.F64, 1e-10, bad_mode, 0, 0, ranks, None, None)
    with pytest.raises(ValueError, match="cutoff_mode"):
        N.check(rc, "ndmps_roundtrip_host")


@pytest.mark.gpu
def test_core_capacity_too_small_is_reported_and_context_recovers():
    import ctypes as C
    from imgcompressionmps import _native as N
    from imgcompressionmps import _ops
    torch = _torch()
    shape, mode = (30, 40, 50), "rsum2"
    d = dense_of(shape, "f64")
    dims = list(d.shape)
    dense = torch.from_numpy(d).cuda()
    caps = [dims[0] * 4, 4 * dims[1] * 50, 50 * dims[2]]             # core 0 can hold rank 4 only
    bufs = [torch.empty(c, dtype=torch.float64, device="cuda") for c in caps]
    ranks = (C.c_int64 * 2)()
    rc = N.load_library().ndmps_ttsvd(N.handle(), N.ptr(dense), N.F64, 3, N.i64_array(dims), 1e-4, N.CUTOFF_MODES[mode],
                                      0, 2, N.ptr_array(bufs), N.i64_array(caps), ranks, None, 0)
    assert rc == -4                                                  # NDMPS_ERR_CAPACITY
    with pytest.raises(N.NativeError, match="capacity"):
        N.check(rc, "ndmps_ttsvd")
    cores, ranks, svals = _ops.ttsvd(dense, dims, cutoff=1e-4, cutoff_mode=mode)
    _check_sweep(cores, ranks, svals, oracle_sweep(shape, "f64", 1e-4, mode, None, 2), "f64")
