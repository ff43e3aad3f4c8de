"""Masked sampling cost on the GPU: the sampling step and the posterior op alone, masked against unmasked.

1. The CUDA-graph sampling step at B = 64 @128x128, bf16, eta = 1 (the configuration bench.py's sampling line runs), masked
   (a feathered ellipse mask) and unmasked, alternated within the run; device events around whole runs, ms per step.
2. The posterior op alone, every form over the same shape, from one d3fk_run call of many launches between two CUDA events.
   The launches cycle through enough buffer sets that their total exceeds the 126 MB L2, so every launch reads HBM.
   Bytes per element: unmasked 12 (x read and written, x0_hat); masked at most 17.33 (plus src and the 1/3-element mask
   read) — less with a hard mask, where a 4-pixel vector of all-0 or all-1 mask reads only the inputs its update needs.
3. A device-to-device copy of 1 GiB as the measured bandwidth peak the kernel shares are quoted against.
Prints the device name and power limit with the numbers.  Needs a B200; there is no CPU path."""
import argparse
import subprocess
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import denoising_diffusion_deep_fake_b200 as d3  # noqa: E402
from denoising_diffusion_deep_fake_b200 import _lib  # noqa: E402
from denoising_diffusion_deep_fake_b200.functional import posterior_coeffs  # noqa: E402
from denoising_diffusion_deep_fake_b200.sampler import Sampler  # noqa: E402

DEV = "cuda:0"


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def ellipse_mask(B, H, W, feather=0.15):
    yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32), indexing="ij")
    d = torch.sqrt(((xx - (W - 1) / 2) / (0.32 * W)) ** 2 + ((yy - (H - 1) / 2) / (0.4 * H)) ** 2)
    m = ((1.0 - d) / feather).clamp(0, 1) if feather > 0 else (d < 1).float()
    return m.expand(B, 1, H, W).contiguous().to(DEV)


def timed(fn, reps=1):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def copy_peak_gbs():
    n = 1 << 28                                    # 1 GiB of float32
    src = torch.empty(n, device=DEV).uniform_()
    dst = torch.empty_like(src)
    dst.copy_(src)
    ms = statistics.median(timed(lambda: dst.copy_(src), 5) for _ in range(5))
    return 2 * 4 * n / (ms * 1e-3) / 1e9


def step_times(B, H, n_steps, rounds):
    torch.manual_seed(0)
    model = d3.Unet(precision="bf16").to(DEV).eval()
    src = torch.randn(B, 3, H, H, device=DEV).clamp(-1, 1)
    mask = ellipse_mask(B, H, H)
    plain = Sampler(model, B, H, H, n_steps, r_start=1.0, eta=1.0, seed=7)
    masked = Sampler(model, B, H, H, n_steps, r_start=1.0, eta=1.0, seed=7, masked=True)
    assert plain.kernels_per_step == masked.kernels_per_step
    runs = {"unmasked": lambda: plain.run(), "masked": lambda: masked.run(src=src, mask=mask)}
    for f in runs.values():
        f()
        f()                                        # capture + warm-up
    out = {k: [] for k in runs}
    for _ in range(rounds):
        for k, f in runs.items():
            out[k].append(timed(f) / n_steps)
    return out, plain.kernels_per_step


def kernel_times(B, H, reps):
    n = B * 3 * H * H
    per_set = 4 * n * 3 + 4 * B * H * H           # x, x0_hat, src, mask
    sets = max(2, -(-3 * 126 * 2 ** 20 // per_set))   # > 3x the L2 in total
    g = torch.Generator(device=DEV).manual_seed(0)
    bufs = [[torch.randn(B, 3, H, H, device=DEV, generator=g) for _ in range(3)] for _ in range(sets)]
    masks = {"hard": ellipse_mask(B, H, H, feather=0), "soft": ellipse_mask(B, H, H),
             "ones": torch.ones(B, 1, H, H, device=DEV), "zeros": torch.zeros(B, 1, H, H, device=DEV)}
    mask_sets = {k: [m.clone() for _ in range(sets)] for k, m in masks.items()}
    k_xi, k_x0, sigma = posterior_coeffs(0.6, 0.55, 1.0)
    _lib.init(0)
    forms = {}
    for name, eta_sigma in (("unmasked", sigma), ("unmasked eta=0", 0.0)):
        forms[name] = [_lib.make_op(_lib.OP_POSTERIOR, n=n, x=x.data_ptr(), x0_hat=h.data_ptr(), k_xi=k_xi, k_x0=k_x0,
                                    sigma=eta_sigma, seed=1, offset=2) for x, h, _ in bufs]
    for mk in masks:
        forms[f"masked {mk}"] = [
            _lib.make_op(_lib.OP_POSTERIOR, n=n, x=x.data_ptr(), x0_hat=h.data_ptr(), k_xi=k_xi, k_x0=k_x0, sigma=sigma,
                         seed=1, offset=2, r_prev=0.55, src=s.data_ptr(), mask=mask_sets[mk][i].data_ptr(),
                         chw=3 * H * H, hw=H * H)
            for i, (x, h, s) in enumerate(bufs)]
    stream = torch.cuda.current_stream().cuda_stream
    lists = {k: _lib.OpList(ops * max(1, reps // sets)) for k, ops in forms.items()}
    for ol in lists.values():
        ol.run(stream)
    res = {k: [] for k in lists}
    for _ in range(5):                             # alternate the forms
        for k, ol in lists.items():
            res[k].append(timed(lambda: ol.run(stream)) / len(ol))
    hard_frac = float((masks["hard"] > 0).float().mean())
    return {k: statistics.median(v) for k, v in res.items()}, n, hard_frac


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=128)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--launches", type=int, default=400)
    a = ap.parse_args()
    print(f"device: {device_info()}")
    peak = copy_peak_gbs()
    print(f"copy peak (1 GiB device-to-device, read + write): {peak:.0f} GB/s")
    ms, n, hard_frac = kernel_times(a.batch, a.size, a.launches)
    print(f"posterior op alone, B={a.batch} @{a.size}x{a.size} ({n / 1e6:.2f} M elements), buffers cycled past L2; "
          f"hard mask: {hard_frac:.1%} of pixels generated")
    bpe = {"unmasked": 12.0, "unmasked eta=0": 12.0, "masked hard": 8.0 + 4.0 * hard_frac + 4.0 / 3,
           "masked soft": 16.0 + 4.0 / 3, "masked ones": 12.0 + 4.0 / 3, "masked zeros": 8.0 + 4.0 / 3}
    for k, t in ms.items():
        gbs = bpe[k] * n / (t * 1e-3) / 1e9
        print(f"  {k:16s} {t * 1e3:7.2f} us  {bpe[k]:5.2f} B/element moved  {gbs:6.0f} GB/s  {gbs / peak:6.1%} of copy peak"
              f"  (17.33 B/element floor: {17.33 * n / (t * 1e-3) / 1e9 / peak:6.1%})")
    st, kps = step_times(a.batch, a.size, a.steps, a.rounds)
    u, m = statistics.median(st["unmasked"]), statistics.median(st["masked"])
    print(f"sampling step, B={a.batch} @{a.size}x{a.size} bf16 eta=1, {kps} kernels/step both, median of {a.rounds} "
          f"alternated runs of {a.steps} steps: unmasked {u:.4f} ms, masked {m:.4f} ms ({(m / u - 1):+.2%}); "
          f"spread unmasked {min(st['unmasked']):.4f}-{max(st['unmasked']):.4f}, "
          f"masked {min(st['masked']):.4f}-{max(st['masked']):.4f}")
    assert _lib.load().d3fk_device_error_flag() == 0


if __name__ == "__main__":
    main()
