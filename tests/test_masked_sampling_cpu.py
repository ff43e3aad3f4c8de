"""Masked (replacement-inpainting) sampling, the parts that need no GPU: the float64 definition (tests/masked_oracle.py),
mask normalisation, the sampler's coefficient table with its r_prev column, the CLI options and the ABI mirror."""
import ctypes
import math

import numpy as np
import pytest
import torch

import oracle
from denoising_diffusion_deep_fake_b200 import _lib
from denoising_diffusion_deep_fake_b200.functional import (noise_ratio_grid, normalize_mask, posterior_coef_table,
                                                           posterior_coeffs)
from masked_oracle import masked_posterior_step, masked_sample_loop

B, H, W, N_STEPS = 2, 8, 12, 6


def toy_model(x):
    """A deterministic stand-in for the U-Net (float64)."""
    return 0.5 * torch.tanh(x) + 0.1 * x.roll(1, dims=-1)


def inputs(eta_noises=True):
    g = torch.Generator().manual_seed(3)
    x_start = torch.randn(B, 3, H, W, generator=g, dtype=torch.float64)
    src = torch.rand(B, 3, H, W, generator=g, dtype=torch.float64) * 2 - 1
    noises = torch.randn(N_STEPS, B, 3, H, W, generator=g, dtype=torch.float64) if eta_noises else None
    known = torch.randn(N_STEPS, B, 3, H, W, generator=g, dtype=torch.float64)
    return x_start, src, noises, known


# ---- oracle -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("eta", [0.0, 1.0])
@pytest.mark.parametrize("r_start", [1.0, 0.6])
def test_oracle_mask_of_ones_is_sample_loop(eta, r_start):
    x_start, src, noises, known = inputs()
    ones = torch.ones(B, 1, H, W, dtype=torch.float64)
    want = oracle.sample_loop(toy_model, x_start, N_STEPS, r_start, eta, noises)
    got = masked_sample_loop(toy_model, x_start, src, ones, N_STEPS, r_start, eta, noises, known)
    assert torch.equal(got, want)


@pytest.mark.parametrize("eta", [0.0, 1.0])
def test_oracle_mask_of_zeros_keeps_the_noised_source(eta):
    x_start, src, noises, known = inputs()
    zeros = torch.zeros(B, 1, H, W, dtype=torch.float64)
    out, traj = masked_sample_loop(toy_model, x_start, src, zeros, N_STEPS, 1.0, eta, noises, known,
                                   return_trajectory=True)
    assert torch.equal(out, src)
    grid = oracle.noise_ratio_grid(N_STEPS, 1.0).tolist()
    for i in range(N_STEPS - 1):
        r = grid[i + 1]
        assert torch.allclose(traj[i], math.sqrt(1 - r) * src + math.sqrt(r) * known[i], rtol=0, atol=1e-14)


def test_oracle_soft_mask_interpolates_each_step():
    x_start, src, noises, known = inputs()
    g = torch.Generator().manual_seed(9)
    m = torch.rand(B, 1, H, W, generator=g, dtype=torch.float64) * 1.4 - 0.2       # values outside [0, 1] are clamped
    x0_hat = toy_model(x_start)
    args = (x_start, x0_hat, 0.8, 0.6)
    full = masked_posterior_step(*args, src, torch.ones_like(m), noises[0], known[0], eta=1.0)
    keep = masked_posterior_step(*args, src, torch.zeros_like(m), noises[0], known[0], eta=1.0)
    soft = masked_posterior_step(*args, src, m, noises[0], known[0], eta=1.0)
    mc = m.clamp(0, 1)
    assert torch.allclose(soft, mc * full + (1 - mc) * keep, rtol=0, atol=1e-14)
    lo, hi = torch.minimum(full, keep), torch.maximum(full, keep)
    assert bool(((soft >= lo - 1e-14) & (soft <= hi + 1e-14)).all())


def test_oracle_single_pass_is_the_composite():
    _, src, _, _ = inputs()
    m = (torch.rand(B, 1, H, W, generator=torch.Generator().manual_seed(1), dtype=torch.float64) > 0.5).double()
    got = masked_sample_loop(toy_model, src, src, m, 1, 0.0)
    assert torch.equal(got, m * toy_model(src) + (1 - m) * src)


# ---- mask normalisation ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(H, W), (1, 1, H, W), (B, 1, H, W)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bool])
def test_normalize_mask_accepts(shape, dtype):
    m = torch.rand(shape, generator=torch.Generator().manual_seed(0)) > 0.5
    m = m.to(dtype) if dtype == torch.bool else m.float() * 0.75
    out = normalize_mask(m, B, H, W)
    assert out.shape == (B, 1, H, W) and out.dtype == torch.float32 and out.is_contiguous()
    assert torch.equal(out, m.to(torch.float32).reshape(-1, 1, H, W).expand(B, 1, H, W))


@pytest.mark.parametrize("shape", [(B, 3, H, W), (B, H, W), (1, H, W), (H, W + 1), (B + 1, 1, H, W), (W, H)])
def test_normalize_mask_rejects_shapes(shape):
    with pytest.raises(ValueError):
        normalize_mask(torch.ones(shape), B, H, W)


@pytest.mark.parametrize("mask", [torch.ones(H, W, dtype=torch.float64), torch.ones(H, W, dtype=torch.uint8),
                                  torch.ones(H, W, dtype=torch.bfloat16), np.ones((H, W), np.float32)])
def test_normalize_mask_rejects_dtypes(mask):
    with pytest.raises(TypeError):
        normalize_mask(mask, B, H, W)


# ---- coefficient table --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_steps,r_start,eta", [(20, 1.0, 0.0), (7, 0.6, 1.0), (1, 1.0, 0.5)])
def test_coef_table_rows(n_steps, r_start, eta):
    grid = noise_ratio_grid(n_steps, r_start)
    rows = posterior_coef_table(grid, eta)
    assert len(rows) == n_steps
    for i, row in enumerate(rows):
        assert row[:3] == posterior_coeffs(grid[i], grid[i + 1], eta)
        assert row[3] == grid[i + 1]
    assert rows[-1] == (0.0, 1.0, 0.0, 0.0)                # the last step returns x0_hat; known = src


def test_coef_table_from_ratio_zero():
    """r_start = 0 (the Sampler's grid of zeros): every step returns x0_hat and composites with the source itself."""
    assert posterior_coef_table([0.0] * 4, 1.0) == [(0.0, 1.0, 0.0, 0.0)] * 3


# ---- ABI and CLI --------------------------------------------------------------------------------------------------
def test_op_size_and_posterior_fields():
    assert ctypes.sizeof(_lib.Op) == 480
    P = _lib.PosteriorParams
    assert P.r_prev.offset == 60                            # the former padding slot after sigma
    assert (P.src.offset, P.mask.offset, P.known_noise.offset, P.chw.offset, P.hw.offset) == (80, 88, 96, 104, 108)
    assert ctypes.sizeof(P) == 112
    assert _lib.load().d3fk_sizeof_op() == 480


def test_cli_sample_lists_source_and_mask():
    from click.testing import CliRunner
    from denoising_diffusion_deep_fake_b200.main import cli
    res = CliRunner().invoke(cli, ["sample", "--help"])
    assert res.exit_code == 0
    assert "--source" in res.output and "--mask" in res.output


def test_cli_sample_source_needs_mask(tmp_path):
    from click.testing import CliRunner
    from denoising_diffusion_deep_fake_b200.main import cli
    res = CliRunner().invoke(cli, ["sample", "--source", str(tmp_path / "src.pt")])
    assert res.exit_code == 2 and "--source and --mask go together" in res.output
