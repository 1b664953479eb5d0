#!/usr/bin/env python
"""tcgen05 paths (csrc/tc_gemm.cu) against float64 references on the B200: accuracy and time.

    python tools/tc_probe.py [gram] [gemm] [sweep]

gram : G = M M^T on bf16x3 planes vs the FP64-tensor-pipe Gram (exact
       float64 accumulation of the same float32 data), on a random and a phantom unfolding.
gemm : the four operand-major combinations and both output orders of gemm_tc vs torch float64.
sweep: one 256^3 / 512^3 volume through NDMPS.from_tensor / to_tensor with the tcgen05 paths on and
       off: bonds, singular values, reconstruction difference, stage times.
torch is the float64 checker here, never the thing measured.
"""
import ctypes as C
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
for p in (str(ROOT), str(ROOT / "img-compression-mps_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

from imgcompressionmps import _native as N, _ops   # noqa: E402


def timed(fn, reps=5):
    fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def gram_case(name, m):
    ctx = N.context()
    ctx.set_option("gram_path", 0)
    ctx.set_option("tc", 0)
    exact = _ops.gram(m)
    t_dmma = timed(lambda: _ops.gram(m))
    lam = torch.linalg.eigvalsh(exact).flip(0)
    ctx.set_option("gram_path", 3)
    g = _ops.gram(m)
    t_tc = timed(lambda: _ops.gram(m))
    err = (g - exact)
    rel_max = float(err.abs().max() / exact.abs().max())
    nz = exact.diagonal() > 0
    rel_diag = float((err.diagonal()[nz].abs() / exact.diagonal()[nz]).max())
    mean_rel_diag = float((err.diagonal()[nz] / exact.diagonal()[nz]).mean())
    lam_tc = torch.linalg.eigvalsh(g).flip(0)
    k = min(64, lam.numel())
    sv_err = float(((lam_tc[:k].clamp_min(0).sqrt() - lam[:k].clamp_min(0).sqrt()).abs() / lam[0].sqrt()).max())
    sym = float((g - g.T).abs().max())
    print(f"  gram {name} {tuple(m.shape)}: tc {t_tc:.3f} ms (dmma {t_dmma:.3f} ms)  max|dG|/max|G| {rel_max:.2e}  "
          f"diag rel max {rel_diag:.2e} mean {mean_rel_diag:+.2e}  top-{k} sigma err / sigma_1 {sv_err:.2e}  asym {sym:.1e}", flush=True)
    ctx.set_option("gram_path", 0)
    ctx.set_option("tc", 1)


def run_gram():
    g = torch.Generator(device="cuda").manual_seed(1)
    for rows, cols in ((512, 32768), (360, 32768), (512, 262144), (2560, 16384)):
        m = torch.rand((rows, cols), device="cuda", generator=g, dtype=torch.float32)
        gram_case("uniform[0,1)", m)
    sys.path.insert(0, str(ROOT))
    from bench import synthetic_volume
    vol = torch.from_numpy(synthetic_volume((256, 256, 256), 2026)).cuda()
    dense = _ops.encode(vol).reshape(512, -1).contiguous()
    gram_case("phantom 256^3 first group", dense)
    # heavy-tailed rows: one element 300x the rest -> rho^2 ~ 9e4 / (1 + ...) > 4096: the device-side flag must hand
    # the matrix to the exact kernel (error 0)
    m = torch.rand((256, 16384), device="cuda", generator=g, dtype=torch.float32)
    m[:, 5] = 2000.0
    gram_case("heavy-tailed rows (exact fallback expected)", m)
    m = torch.randn((512, 32768), device="cuda", generator=g, dtype=torch.float32) * torch.logspace(0, -6, 512, device="cuda")[:, None].float()
    gram_case("gaussian rows, norms over 6 decades", m)


def gemm_ref(a, b):
    return a.double() @ b.double()


def call_gemm(a, b, out_dtype, out_t):
    m, k = a.shape
    _, n = b.shape
    c = torch.empty((n, m) if out_t else (m, n), dtype=out_dtype, device="cuda")
    ctx = N.context()
    ctx.set_option("gemm_out_t", 1 if out_t else 0)
    try:
        N.check(N.load_library().ndmps_gemm(N.handle(), m, n, k, 1.0, N.ptr(a), N.dtype_code(a.dtype), a.stride(0), a.stride(1),
                                            N.ptr(b), N.dtype_code(b.dtype), b.stride(0), b.stride(1), N.ptr(c),
                                            N.dtype_code(out_dtype), m if out_t else n), "ndmps_gemm")
    finally:
        ctx.set_option("gemm_out_t", 0)
    return c.T if out_t else c


def run_gemm():
    ctx = N.context()
    g = torch.Generator(device="cuda").manual_seed(2)
    cases = [  # (m, n, k, a_mn, b_mn, out_t, dtype_a, dtype_b, label)
        (32768, 64, 512, True, False, True, torch.float32, torch.float64, "projection T = P^T M (A MN-major, out transposed)"),
        (262144, 64, 512, True, False, True, torch.float32, torch.float64, "projection at 512^3"),
        (4096, 45, 360, True, False, True, torch.float32, torch.float64, "projection, ragged (n = 45, k = 360)"),
        (4096, 4096, 64, False, True, False, torch.float32, torch.float32, "contraction dense = X W (B MN-major)"),
        (32768, 4096, 64, False, True, False, torch.float32, torch.float32, "contraction at 512^3"),
        (1000, 200, 136, False, True, False, torch.float32, torch.float32, "ragged row-major"),
        (640, 128, 320, False, False, False, torch.float32, torch.float32, "both K-major"),
        (640, 72, 200, True, True, False, torch.float64, torch.float64, "both MN-major, float64 in"),
        (16384, 128, 1024, True, False, True, torch.float32, torch.float64, "chi = 128 projection"),
    ]
    for m, n, k, a_mn, b_mn, out_t, da, db, label in cases:
        a = (torch.rand((k, m) if a_mn else (m, k), device="cuda", generator=g, dtype=torch.float64) - 0.3).to(da)
        b = (torch.rand((k, n) if b_mn else (n, k), device="cuda", generator=g, dtype=torch.float64) - 0.5).to(db)
        av = a.T if a_mn else a
        bv = b if b_mn else b.T
        want = gemm_ref(av, bv)
        ctx.set_option("gemm_path", 3)
        got = call_gemm(av, bv, torch.float32, out_t)
        t_tc = timed(lambda: call_gemm(av, bv, torch.float32, out_t), 3)
        ctx.set_option("gemm_path", 0)
        ctx.set_option("tc", 0)
        base = _ops.gemm(av, bv, out_dtype=torch.float32)
        t_base = timed(lambda: _ops.gemm(av, bv, out_dtype=torch.float32), 3)
        ctx.set_option("tc", 1)
        scale = float(want.abs().max())
        e_tc = float((got.double() - want).abs().max()) / scale
        e_base = float((base.double() - want).abs().max()) / scale
        print(f"  gemm {label}: m {m} n {n} k {k}: tc {t_tc:.3f} ms err {e_tc:.2e} | current path {t_base:.3f} ms err {e_base:.2e}", flush=True)


def run_sweep():
    sys.path.insert(0, str(ROOT))
    from bench import synthetic_volume
    from imgcompressionmps.core.ndmps import NDMPS
    ctx = N.context()
    for n, seed in ((256, 2026), (512, 2027)):
        vol = torch.from_numpy(synthetic_volume((n, n, n), seed)).cuda()
        res = {}
        for tc in (0, 1):
            ctx.set_option("tc", tc)
            obj = NDMPS.from_tensor(vol, max_bond=64)
            rec = obj.to_tensor_device()
            ctx.profile(True)
            ctx.stage_times(reset=True)
            t0 = time.perf_counter()
            for _ in range(3):
                o2 = NDMPS.from_tensor(vol, max_bond=64)
                o2.to_tensor_device()
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) / 3 * 1e3
            st = ctx.stage_times(reset=True)
            ctx.profile(False)
            res[tc] = (obj, rec)
            print(f"  sweep {n}^3 tc={tc}: {ms:.2f} ms/volume  bonds {obj.bond_sizes()}  stages " +
                  " ".join(f"{k}={v[0] / 3:.2f}" for k, v in st.items() if v[1]), flush=True)
        (o0, r0), (o1, r1) = res[0], res[1]
        sv = max(float(np.abs(a - b).max() / b[0]) for a, b in zip(o1.singular_values, o0.singular_values))
        rel = float(torch.linalg.vector_norm((r1 - r0).double()) / torch.linalg.vector_norm(r0.double()))
        print(f"  sweep {n}^3: bonds equal {o0.bond_sizes() == o1.bond_sizes()}  max sigma diff / sigma_1 {sv:.2e}  rec rel diff {rel:.2e}", flush=True)
    ctx.set_option("tc", 1)


if __name__ == "__main__":
    what = sys.argv[1:] or ["gram", "gemm"]
    if "gram" in what:
        run_gram()
    if "gemm" in what:
        run_gemm()
    if "sweep" in what:
        run_sweep()
