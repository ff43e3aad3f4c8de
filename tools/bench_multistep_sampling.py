"""Second-order multistep (DPM-Solver++ 2M) sampling on the GPU: its cost per step and what it buys per step.

1. The CUDA-graph sampling step at B = 64 @128x128, bf16, eta = 0, first-order posterior against 2M (both on the logsnr
   grid, so the 2M steps are second order), alternated within the run; device events around whole runs, ms per step.
2. The 2M op alone against its bytes: 20 B/element (x read and written, x0_hat read, x0_prev read and written) with
   c != 0, 16 B with c = 0; the first-order op (12 B) beside it.  One d3fk_run call of many launches between two CUDA
   events, cycling through enough buffer sets that their total exceeds the 126 MB L2, so every launch reads HBM.  A 1 GiB
   device-to-device copy is the measured bandwidth peak the shares are quoted against.
3. Accuracy against steps on the product in fp32 with trained weights (oracle.short_training_run, 150 steps + BatchNorm
   calibration, as the tests' fixture): PSNR of each solver and grid at N = 5, 10, 20, 40 against a 400-step float64 2M
   oracle run on the same grid, B = 4 @64x64, eta = 0, r_start 1 and 0.6.
Prints the device name and power limit with the numbers.  Needs a B200; there is no CPU path."""
import argparse
import copy
import math
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import denoising_diffusion_deep_fake_b200 as d3  # noqa: E402
import oracle  # noqa: E402
from denoising_diffusion_deep_fake_b200 import _lib  # noqa: E402
from denoising_diffusion_deep_fake_b200.functional import dpmpp_2m_coeffs, noise_ratio_grid  # noqa: E402
from denoising_diffusion_deep_fake_b200.sampler import Sampler  # noqa: E402
from bench_masked_sampling import copy_peak_gbs, device_info, timed  # noqa: E402
from multistep_oracle import dpmpp_2m_sample_loop  # noqa: E402

DEV = "cuda:0"


def step_times(B, H, n_steps, rounds):
    torch.manual_seed(0)
    model = d3.Unet(precision="bf16").to(DEV).eval()
    smp = {s: Sampler(model, B, H, H, n_steps, r_start=1.0, eta=0.0, seed=7, solver=s, schedule="logsnr")
           for s in ("posterior", "dpmpp_2m")}
    assert smp["posterior"].kernels_per_step == smp["dpmpp_2m"].kernels_per_step
    for s in smp.values():
        s.run()
        s.run()                                    # capture + warm-up
    out = {k: [] for k in smp}
    for _ in range(rounds):
        for k, s in smp.items():
            out[k].append(timed(s.run) / n_steps)
    return out, smp["posterior"].kernels_per_step


def kernel_times(B, H, reps):
    n = B * 3 * H * H
    sets = max(2, -(-3 * 126 * 2 ** 20 // (4 * n * 3)))   # > 3x the L2 in total
    g = torch.Generator(device=DEV).manual_seed(0)
    bufs = [[torch.randn(B, 3, H, H, device=DEV, generator=g) for _ in range(3)] for _ in range(sets)]
    k_xi, k_x0, sigma, c = dpmpp_2m_coeffs(0.7, 0.6, 0.55, 0.0)
    _lib.init(0)
    forms = {"posterior (12 B)": [_lib.make_op(_lib.OP_POSTERIOR, n=n, x=x.data_ptr(), x0_hat=h.data_ptr(), k_xi=k_xi,
                                               k_x0=k_x0, sigma=sigma) for x, h, _ in bufs]}
    for name, cc in (("2M c != 0 (20 B)", c), ("2M c = 0 (16 B)", 0.0)):
        forms[name] = [_lib.make_op(_lib.OP_POSTERIOR_2M, x0_prev=p.data_ptr(), c=cc,
                                    base=dict(n=n, x=x.data_ptr(), x0_hat=h.data_ptr(), k_xi=k_xi, k_x0=k_x0, sigma=sigma))
                       for x, h, p in bufs]
    stream = torch.cuda.current_stream().cuda_stream
    lists = {k: _lib.OpList(ops * max(1, reps // sets)) for k, ops in forms.items()}
    for ol in lists.values():
        ol.run(stream)
    res = {k: [] for k in lists}
    for _ in range(5):                             # alternate the forms
        for k, ol in lists.items():
            res[k].append(timed(lambda: ol.run(stream)) / len(ol))
    return {k: statistics.median(v) for k, v in res.items()}, n


def psnr(a, b):
    mse = ((a.double() - b.double()) ** 2).mean().item()
    return 10 * math.log10((b.max() - b.min()).item() ** 2 / max(mse, 1e-30))


def quality_table(steps_list):
    torch.manual_seed(0)
    ref = oracle.Unet()
    sd = oracle.short_training_run(ref, copy.deepcopy(ref.state_dict()), steps=150, device=DEV, dtype=torch.float64,
                                   calibrate=30)
    sd = {k: v.cpu() for k, v in sd.items()}
    r64 = copy.deepcopy(ref)
    r64.load_state_dict(sd)
    r64 = r64.double().to(DEV).eval()
    model = d3.Unet(precision="fp32")
    model.load_state_dict(sd)
    model = model.to(DEV).eval()
    B, H = 4, 64
    g = torch.Generator(device=DEV).manual_seed(5)
    src = (torch.nn.functional.avg_pool2d(0.5 * torch.randn(B, 3, H, H, generator=g, device=DEV), 5, 1, 2) * 2.5).clamp(-1, 1)
    noise = torch.randn(B, 3, H, H, generator=g, device=DEV)
    for r0 in (1.0, 0.6):
        x = math.sqrt(1.0 - r0) * src + math.sqrt(r0) * noise
        for kind in ("linear", "logsnr"):
            fine = dpmpp_2m_sample_loop(r64, x.double(), noise_ratio_grid(400, r0, kind=kind), 0.0)
            cells = []
            for n in steps_list:
                p = [psnr(Sampler(model, B, H, H, n, r_start=r0, solver=s, schedule=kind).run(x), fine)
                     for s in ("posterior", "dpmpp_2m")]
                cells.append(f"{p[0]:.1f} / {p[1]:.1f}")
            print(f"| {r0}, {kind}: first order / 2M | " + " | ".join(cells) + " |", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=128)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--launches", type=int, default=400)
    ap.add_argument("--skip-quality", action="store_true")
    a = ap.parse_args()
    print(f"device: {device_info()}")
    peak = copy_peak_gbs()
    print(f"copy peak (1 GiB device-to-device, read + write): {peak:.0f} GB/s")
    ms, n = kernel_times(a.batch, a.size, a.launches)
    print(f"posterior ops alone, B={a.batch} @{a.size}x{a.size} ({n / 1e6:.2f} M elements), buffers cycled past L2")
    for k, t in ms.items():
        bpe = float(k.split("(")[1].split()[0])
        gbs = bpe * n / (t * 1e-3) / 1e9
        print(f"  {k:18s} {t * 1e3:7.2f} us  {gbs:6.0f} GB/s  {gbs / peak:6.1%} of copy peak "
              f"(byte floor at that peak {bpe * n / (peak * 1e9) * 1e6:6.2f} us)")
    st, kps = step_times(a.batch, a.size, a.steps, a.rounds)
    p, m = statistics.median(st["posterior"]), statistics.median(st["dpmpp_2m"])
    print(f"sampling step, B={a.batch} @{a.size}x{a.size} bf16 eta=0 logsnr, {kps} kernels/step both, median of "
          f"{a.rounds} alternated runs of {a.steps} steps: posterior {p:.4f} ms, 2M {m:.4f} ms ({(m / p - 1):+.2%}); "
          f"spread posterior {min(st['posterior']):.4f}-{max(st['posterior']):.4f}, "
          f"2M {min(st['dpmpp_2m']):.4f}-{max(st['dpmpp_2m']):.4f}")
    assert _lib.load().d3fk_device_error_flag() == 0
    if not a.skip_quality:
        steps_list = (5, 10, 20, 40)
        print("PSNR against a 400-step float64 2M oracle run on the same grid (fp32 product, trained weights, B=4 @64x64, "
              "eta 0)")
        print("| r_start, grid | " + " | ".join(f"N = {n}" for n in steps_list) + " |")
        quality_table(steps_list)


if __name__ == "__main__":
    main()
