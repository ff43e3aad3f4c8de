"""Timings of the autograd modes of d3fk.Unet (bf16 engine), one JSON line on stdout:

- eval forward under no_grad (the fused eval plan) vs eval forward + backward on the frozen-BN plan, without and with the
  input gradient, at the sampling shape (B = 64 @ 128^2) and the training shape (B = 256 @ 64^2);
- the training step (forward + backward) without and with the input gradient (B = 256 @ 64^2);
- the stem input-gradient kernel (stem_dgrad.cu) vs the generic tensor-core mode-1 gather on the same operands (steered
  there by a zero bias, which the dedicated kernel does not take);
- the frozen single-pass BatchNorm backward on the three largest BN tensors of the B = 256 @ 64^2 step against its HBM floor
  (dy and x read, dx written, mask from x: 6 bytes per element at 7.7 TB/s).

Times are CUDA-event medians over repeated runs after a warm-up; nothing is written to the repository tree.
Usage: python tools/bench_grad_modes.py [--reps 20]"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import denoising_diffusion_deep_fake_b200 as d3          # noqa: E402
from denoising_diffusion_deep_fake_b200 import _lib       # noqa: E402

DEV = "cuda:0"
HBM_BPS = 7.7e12


def timed(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return round(ts[len(ts) // 2], 4)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name(0)
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0)


def model_modes(reps):
    torch.manual_seed(0)
    m = d3.Unet(precision="bf16").to(DEV)
    res = {}
    for B, H in ((64, 128), (256, 64)):
        x = torch.randn(B, 3, H, H, device=DEV).clamp(-1, 1)
        dy = torch.randn_like(x)
        m.eval()

        def fwd_nograd():
            with torch.no_grad():
                m(x)

        def fwd_bwd(want_dx):
            def f():
                xi = x.detach().requires_grad_(want_dx)
                m(xi).backward(dy)
            return f

        key = f"B{B}_{H}"
        res[f"eval_fwd_nograd_ms_{key}"] = timed(fwd_nograd, reps)
        res[f"eval_fwd_bwd_ms_{key}"] = timed(fwd_bwd(False), reps)
        res[f"eval_fwd_bwd_dx_ms_{key}"] = timed(fwd_bwd(True), reps)
        if B == 256:
            m.train()
            res[f"train_step_ms_{key}"] = timed(fwd_bwd(False), reps)
            res[f"train_step_dx_ms_{key}"] = timed(fwd_bwd(True), reps)
    return res


def stem_dgrad(reps):
    B, H, W = 256, 64, 64
    dy = torch.randn(B, H // 2, W // 2, 64, device=DEV).to(torch.bfloat16)
    w = torch.randn(3, 49 * 64, device=DEV).to(torch.bfloat16)
    out = torch.empty(B, 3, H, W, device=DEV)
    zero_bias = torch.zeros(3, device=DEV)
    f = dict(dtype=_lib.BF16, mode=1, src0=dy.data_ptr(), c0=64, ld0=64, B=B, Hi=H // 2, Wi=W // 2, Ho=H, Wo=W, kh=7, kw=7,
             stride=2, pad=3, w=w.data_ptr(), Cout=3, out_nchw=out.data_ptr())
    s = torch.cuda.current_stream().cuda_stream
    dedicated = _lib.OpList([_lib.make_op(_lib.OP_CONV, **f)])
    generic = _lib.OpList([_lib.make_op(_lib.OP_CONV, shift=zero_bias.data_ptr(), **f)])
    n0 = _lib.launch_count()
    t_d = timed(lambda: dedicated.run(s), reps)
    y_d = out.clone()
    try:
        t_g = timed(lambda: generic.run(s), reps)
        same = bool(torch.allclose(out, y_d, rtol=1e-5, atol=1e-3))
    except _lib.D3fkError as e:
        t_g, same = float("nan"), str(e)
    floor_us = (dy.numel() * 2 + out.numel() * 4) / HBM_BPS * 1e6
    return {"stem_dgrad_us_B256_64": round(t_d * 1e3, 2), "stem_dgrad_generic_us_B256_64": round(t_g * 1e3, 2),
            "stem_dgrad_hbm_floor_us": round(floor_us, 2), "stem_dgrad_generic_agrees": same,
            "stem_dgrad_launches": _lib.launch_count() - n0}


def frozen_bn(reps):
    out = {}
    for name, C, count in (("stem", 64, 256 * 32 * 32), ("dec4", 16, 256 * 64 * 64), ("dec3", 32, 256 * 32 * 32)):
        x = torch.randn(count, C, device=DEV).to(torch.bfloat16)
        dy = torch.randn(count, C, device=DEV).to(torch.bfloat16)
        dx = torch.empty_like(x)
        vec = lambda v: torch.full((C,), v, device=DEV)
        gamma, mean, invstd, scale, shift = vec(1.0), vec(0.0), vec(1.0), vec(1.0), vec(0.0)
        bstats = torch.zeros(2, C, dtype=torch.float64, device=DEV)
        dg, db = vec(0.0), vec(0.0)
        op = _lib.make_op(_lib.OP_BN_BWD, dtype=_lib.BF16, C=C, relu=1, mask_from_x=1, count=count, x=x.data_ptr(), ldx=C,
                          gamma=gamma.data_ptr(), mean=mean.data_ptr(), invstd=invstd.data_ptr(), scale=scale.data_ptr(),
                          shift=shift.data_ptr(), dy=dy.data_ptr(), lddy=C, dx=dx.data_ptr(), lddx=C, bstats=bstats.data_ptr(),
                          dgamma=dg.data_ptr(), dbeta=db.data_ptr(), frozen=1)
        ol = _lib.OpList([op])
        s = torch.cuda.current_stream().cuda_stream
        t = timed(lambda: ol.run(s), reps)
        floor_us = count * C * 6 / HBM_BPS * 1e6
        out[f"frozen_bn_bwd_us_{name}"] = round(t * 1e3, 2)
        out[f"frozen_bn_bwd_floor_us_{name}"] = round(floor_us, 2)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_grad_modes: needs a B200; there is no CPU measurement")
    _lib.init(0)
    res = {"gpu": gpu_info()}
    res.update(model_modes(a.reps))
    res.update(stem_dgrad(max(a.reps, 50)))
    res.update(frozen_bn(max(a.reps, 50)))
    res["device_error_flag"] = int(_lib.load().d3fk_device_error_flag())
    print(json.dumps(res))


if __name__ == "__main__":
    main()
