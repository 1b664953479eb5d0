"""Device-time probe of the building blocks (CUDA events, warm-up, L2-sized inputs).
Run on the GPU box:  python tools/perf_probe.py [what ...]"""
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "img-compression-mps_b200"))
sys.path.insert(0, str(ROOT))
from imgcompressionmps import _native, _ops  # noqa: E402


def timeit(fn, reps=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    t = sorted(a.elapsed_time(b) for a, b in ev)
    return t[len(t) // 2]


def main(which):
    torch.cuda.set_device(0)
    ctx = _native.context()
    g = torch.Generator(device="cuda").manual_seed(0)
    if "eigh" in which:
        for n in (8, 64, 128, 256, 512, 1024):
            a = torch.randn(n, 4 * n, dtype=torch.float64, device="cuda", generator=g)
            gm = a @ a.T
            try:
                ms = timeit(lambda: _ops.eigh(gm), reps=3, warm=1)
                _, _, sw = _ops.eigh(gm)
                print(f"eigh n={n}: {ms:.3f} ms, {sw} sweeps", flush=True)
            except Exception as exc:
                print(f"eigh n={n}: FAILED {exc}", flush=True)
    if "topk" in which:
        from bench import synthetic_volume
        vol = torch.from_numpy(synthetic_volume((128, 128, 128), 7)).cuda().double()
        cases = []
        for n in (256, 360, 512, 1024, 1536, 2560):
            a = torch.randn(n, 4 * n, dtype=torch.float64, device="cuda", generator=g)
            cases.append((f"random n={n}", a @ a.T))
            m = vol.reshape(-1)[: (vol.numel() // n) * n].reshape(n, -1)
            cases.append((f"volume unfolding n={n}", m @ m.T))
            w = torch.linalg.qr(torch.randn(n, n, dtype=torch.float64, device="cuda", generator=g))[0]
            lam = torch.cat([torch.full((20,), 3.0), torch.full((20,), 3.0 - 1e-13), torch.logspace(0, -6, n - 40)]).double().cuda()
            cases.append((f"clustered n={n}", (w * lam) @ w.T))
        for name, gm in cases:
            n = gm.shape[0]
            k = 64
            gm = 0.5 * (gm + gm.T)
            try:
                ctx.set_option("topk_cluster", 0)
                ms_grid = timeit(lambda: _ops.eigh_topk(gm, k), reps=3, warm=1)
                ctx.set_option("topk_cluster", 1)
                ev, vec, tr, health = _ops.eigh_topk(gm, k)
                ms = timeit(lambda: _ops.eigh_topk(gm, k), reps=3, warm=1)
                name += f" (grid-barrier variant {ms_grid:.3f} ms, cluster launches {int(ctx.stat('cluster_launches'))})"
            except Exception as exc:
                print(f"topk {name}: FAILED {exc}", flush=True)
                continue
            ref = torch.linalg.eigvalsh(gm).flip(0)
            rel = ((ev - ref[:k]).abs() / ref[0]).max().item()
            orth = (vec.T @ vec - torch.eye(k, dtype=torch.float64, device="cuda")).abs().max().item()
            res = ((gm @ vec - vec * ev).norm(dim=0) / ref[0]).max().item()
            print(f"topk {name}: {ms:.3f} ms  health={health} |dlam|/lam1={rel:.2e} orth={orth:.2e} resid={res:.2e} "
                  f"trace err={(tr - ref.sum().item()) / ref.sum().item():.1e}", flush=True)
    if "gram" in which:
        for rows, cols in ((8, 1 << 21), (64, 1 << 18), (512, 1 << 15), (512, 1 << 12), (512, 512), (512, 1 << 18)):
            m = torch.randn(rows, cols, dtype=torch.float32, device="cuda", generator=g)
            ms = timeit(lambda: _ops.gram(m, 0))
            fl = 2.0 * rows * rows * cols
            print(f"gram {rows}x{cols}: {ms:.3f} ms, {fl / ms / 1e9:.2f} TFLOP/s (fp32-equivalent), "
                  f"{rows * cols * 4 / ms / 1e6:.1f} GB/s read", flush=True)
    if "proj" in which:
        for r, rows, cols in ((64, 512, 1 << 15), (64, 512, 1 << 18), (8, 8, 1 << 21)):
            p = torch.randn(rows, r, dtype=torch.float64, device="cuda", generator=g)
            m = torch.randn(rows, cols, dtype=torch.float32, device="cuda", generator=g)
            pt = p.t().contiguous()                      # the sweep makes P^T explicit (row-major) before the big product
            ms = timeit(lambda: _ops.gemm(pt, m, out_dtype=torch.float32))
            print(f"project {r}x{rows} . {rows}x{cols}: {ms:.3f} ms, {2.0 * r * rows * cols / ms / 1e9:.2f} TFLOP/s", flush=True)
    if "permute" in which:
        for shape in ((256, 256, 256), (512, 512, 512), (64, 64, 32, 400)):
            x = torch.randn(shape, dtype=torch.float32, device="cuda", generator=g)
            ms = timeit(lambda: _ops.encode(x))
            d = _ops.encode(x)
            ms2 = timeit(lambda: _ops.decode(d, shape))
            nb = x.numel() * 8
            print(f"permute {shape}: encode {ms:.3f} ms ({nb / ms / 1e6:.0f} GB/s), decode {ms2:.3f} ms ({nb / ms2 / 1e6:.0f} GB/s)", flush=True)
    if "ssim" in which:
        for shape in ((256, 256, 256), (64, 64, 32, 100)):
            a = torch.rand(shape, dtype=torch.float32, device="cuda", generator=g)
            b = a + 0.05 * torch.randn(shape, dtype=torch.float32, device="cuda", generator=g)
            ms = timeit(lambda: _ops.ssim(a, b), reps=3, warm=1)
            print(f"ssim {shape}: {ms:.3f} ms ({a.numel() * 16 / ms / 1e6:.0f} GB/s algorithmic)", flush=True)
            ms = timeit(lambda: _ops.psnr_terms(a, b), reps=3, warm=1)
            print(f"psnr {shape}: {ms:.3f} ms ({a.numel() * 8 / ms / 1e6:.0f} GB/s)", flush=True)
    if "configs" in which:
        from imgcompressionmps.core.ndmps import NDMPS
        from imgcompressionmps.utils.metrics import compute_psnr, compute_ssim_by_dim
        cases = [("cfg4 fMRI subject (64,64,32,400) Std", (64, 64, 32, 400), "Std"),
                 ("cfg5-B video chunk (1920,1080,64) DCT", (1920, 1080, 64), "DCT"),
                 ("cfg1 image (256,256) Std chi=32", (256, 256), "Std")]
        for name, shape, mode in cases:
            x = torch.rand(shape, dtype=torch.float32, device="cuda", generator=g)
            x = x * 0.1 + torch.linspace(0, 1, shape[-1], device="cuda").expand(shape)
            chi = 32 if len(shape) == 2 else 64
            run = lambda: NDMPS.from_tensor(x, mode=mode, max_bond=chi).to_tensor_device()
            run(); run()
            ctx.profile(True); ctx.stage_times(reset=True)
            ms = timeit(run, reps=3, warm=1)
            st = {k: round(v[0] / 4, 3) for k, v in ctx.stage_times().items() if v[1]}
            ctx.profile(False)
            rec = run()
            t_ssim = timeit(lambda: compute_ssim_by_dim(rec, x), reps=3, warm=1) if len(shape) <= 4 else float("nan")
            t_psnr = timeit(lambda: compute_psnr(rec, x), reps=3, warm=1)
            print(f"{name}: encode+sweep+reconstruct {ms:.2f} ms ({x.numel() / ms / 1e6:.2f} Gvoxel/s) stages {st}; "
                  f"SSIM {t_ssim:.2f} ms, PSNR {t_psnr:.2f} ms", flush=True)
    if "stages" in which or "stages512" in which:
        from imgcompressionmps.core.ndmps import NDMPS
        from bench import synthetic_volume
        for n in ((512,) if "stages512" in which else (256,)):
            x = torch.from_numpy(synthetic_volume((n, n, n), 2026)).cuda()
            for _ in range(2):
                NDMPS.from_tensor(x, max_bond=64).to_tensor_device()
            ctx.profile(True)
            ctx.stage_times(reset=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            NDMPS.from_tensor(x, max_bond=64).to_tensor_device()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            print(f"stages {n}^3 chi=64: wall {dt * 1e3:.2f} ms", {k: (round(v[0], 3), v[1]) for k, v in ctx.stage_times().items()}, flush=True)
            ctx.profile(False)


if __name__ == "__main__":
    main(sys.argv[1:] or ["eigh", "gram", "proj", "permute", "ssim", "stages"])
