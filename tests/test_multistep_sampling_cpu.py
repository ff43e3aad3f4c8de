"""Second-order multistep (DPM-Solver++ 2M) sampling, the parts that need no GPU: the coefficient rows and their c = 0
rules, the log-SNR grid, the convergence order of the float64 definition (tests/multistep_oracle.py), the ABI mirror and
the CLI options."""
import ctypes
import math

import pytest
import torch

from denoising_diffusion_deep_fake_b200 import _lib
from denoising_diffusion_deep_fake_b200.functional import (dpmpp_2m_coef_table, dpmpp_2m_coeffs, log_snr,
                                                           noise_ratio_grid, posterior_coef_table, posterior_coeffs)
from multistep_oracle import dpmpp_2m_sample_loop, lam, logsnr_grid

GRIDS = [("linear", 10, 1.0), ("linear", 7, 0.6), ("logsnr", 10, 1.0), ("logsnr", 20, 0.6), ("logsnr", 2, 1.0),
         ("logsnr", 5, 0.3)]


def grid_of(kind, n, r0):
    return noise_ratio_grid(n, r0, kind=kind)


def close(a, b, rel=1e-12):
    return abs(a - b) <= rel * max(abs(a), abs(b), 1e-300)


# ---- coefficient rows ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("eta", [0.0, 1.0])
@pytest.mark.parametrize("kind,n,r0", GRIDS)
def test_rows_are_first_order_at_eta_0_and_1(kind, n, r0, eta):
    grid = grid_of(kind, n, r0)
    for i in range(n):
        got = dpmpp_2m_coeffs(grid[i - 1] if i else None, grid[i], grid[i + 1], eta)[:3]
        want = posterior_coeffs(grid[i], grid[i + 1], eta)
        if grid[i] == 1.0 and eta == 1.0:
            # exactly 0; posterior_coeffs forms it as sqrt(r_prev - sigma^2) and is left with the root of a rounding error
            assert got[0] == 0.0 and abs(want[0]) < 1e-7
            got, want = got[1:], want[1:]
        for g, w in zip(got, want):
            assert close(g, w), (kind, n, r0, eta, i, got, want)


@pytest.mark.parametrize("eta", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("kind,n,r0", GRIDS)
def test_table_c_column(kind, n, r0, eta):
    grid = grid_of(kind, n, r0)
    rows = dpmpp_2m_coef_table(grid, eta)
    assert len(rows) == n and all(len(r) == 5 for r in rows)
    assert rows[0][4] == 0.0                                        # the first step
    assert rows[-1] == (0.0, 1.0, 0.0, 0.0, 0.0)                    # the step to 0 returns x0_hat
    for i in range(1, n - 1):
        h, h_before = lam(grid[i + 1]) - lam(grid[i]), lam(grid[i]) - lam(grid[i - 1])
        if math.isinf(h) or math.isinf(h_before):
            assert rows[i][4] == 0.0                                # the step from r = 1 and the step after it
        else:
            assert close(rows[i][4], h / (2.0 * h_before))
    if r0 == 1.0 and n >= 2:
        assert rows[1][4] == 0.0
    for i, row in enumerate(rows):
        assert row[3] == max(grid[i + 1], 0.0)                      # r_prev: the masked update's known ratio
    if eta in (0.0, 1.0):                                           # the first four columns are today's table
        for i, (row, old) in enumerate(zip(rows, posterior_coef_table(grid, eta))):
            if grid[i] == 1.0 and eta == 1.0:                       # k_xi: see the test above
                assert row[0] == 0.0 and abs(old[0]) < 1e-7
                row, old = row[1:4], old[1:]
            assert all(close(a, b) for a, b in zip(row[:4], old))


def test_rows_at_the_ends():
    # from r = 1 with eta > 0: (0, alpha_t, s_t); eta = 0: (s_t, alpha_t, 0)
    r_t = 0.3
    assert dpmpp_2m_coeffs(None, 1.0, r_t, 0.7) == (0.0, math.sqrt(1 - r_t), math.sqrt(r_t), 0.0)
    assert dpmpp_2m_coeffs(None, 1.0, r_t, 0.0) == (math.sqrt(r_t), math.sqrt(1 - r_t), 0.0, 0.0)
    assert dpmpp_2m_coeffs(1.0, 0.5, 0.2, 0.0)[3] == 0.0           # h_before infinite
    assert dpmpp_2m_coeffs(0.8, 0.5, 0.0, 1.0) == (0.0, 1.0, 0.0, 0.0)   # to r = 0
    assert dpmpp_2m_coef_table([0.0] * 5, 1.0) == [(0.0, 1.0, 0.0, 0.0, 0.0)] * 4
    # general eta: k-diffusion's dpmpp_2m_sde (midpoint) written in r
    r_b, r_i, r_t, eta = 0.7, 0.5, 0.2, 0.5
    h, hb = log_snr(r_t) - log_snr(r_i), log_snr(r_i) - log_snr(r_b)
    k_xi, k_x0, sigma, c = dpmpp_2m_coeffs(r_b, r_i, r_t, eta)
    assert close(k_xi, math.sqrt(r_t / r_i) * math.exp(-eta * h))
    assert close(k_x0, math.sqrt(1 - r_t) * (1 - math.exp(-(1 + eta) * h)))
    assert close(sigma, math.sqrt(r_t) * math.sqrt(1 - math.exp(-2 * eta * h)))
    assert close(c, h / (2 * hb))


# ---- grid ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,r0,r_min", [(2, 1.0, 1e-3), (3, 1.0, 1e-3), (10, 1.0, 1e-3), (20, 0.6, 1e-3), (40, 0.6, 0.01),
                                        (7, 0.999, 1e-3), (5, 0.3, 0.2)])
def test_logsnr_grid(n, r0, r_min):
    grid = noise_ratio_grid(n, r0, kind="logsnr", r_min=r_min)
    assert len(grid) == n + 1 and grid[0] == r0 and grid[-1] == 0.0
    assert all(a > b for a, b in zip(grid, grid[1:]))
    assert abs(grid[-2] - r_min) <= 1e-12 * r_min
    la, lb = lam(min(r0, 1 - r_min)), lam(r_min)
    for k in range(1, n):
        assert abs(lam(grid[k]) - (la + (lb - la) * k / (n - 1))) <= 1e-12 * max(1.0, abs(lb - la))
    assert grid == logsnr_grid(n, r0, r_min)


def test_logsnr_grid_small_and_errors():
    assert noise_ratio_grid(1, 1.0, kind="logsnr") == [1.0, 0.0]
    assert noise_ratio_grid(1, 5e-4, kind="logsnr") == [5e-4, 0.0]          # one step: no interior point
    assert noise_ratio_grid(2, 1.0, kind="logsnr") == [1.0, pytest.approx(1e-3, rel=1e-12), 0.0]
    assert noise_ratio_grid(3, 0.0, kind="logsnr") == [0.0] * 4
    with pytest.raises(ValueError):
        noise_ratio_grid(4, 1e-3, kind="logsnr")                              # 0 < r_start <= r_min
    with pytest.raises(ValueError):
        noise_ratio_grid(4, 5e-4, kind="logsnr")
    for r_min in (0.0, -1e-3, 0.5, 0.7):
        with pytest.raises(ValueError):
            noise_ratio_grid(4, 1.0, kind="logsnr", r_min=r_min)
    with pytest.raises(ValueError):
        noise_ratio_grid(0, 1.0, kind="logsnr")
    with pytest.raises(ValueError):
        noise_ratio_grid(4, 1.0, kind="cosine")
    assert noise_ratio_grid(4, 0.8) == [0.8 * (1 - i / 4) for i in range(5)]  # the linear grid is today's


# ---- order of the float64 definition -------------------------------------------------------------------------------
def test_oracle_convergence_order():
    """A smooth, noise-level-blind denoiser x0_hat = tanh(A x + b) (A, b fixed per pixel) in float64, r_start = 0.9, eta 0,
    the logsnr grid; the error at N = 40 and N = 80 steps against a 2560-step 2M solution gives the empirical order
    log2(e_40/e_80).  Measured: 2M 1.96 (1.86 from 20 to 40), first order 1.03.  A wrong c (its sign, the factor 2, the
    h ratio inverted) drops 2M to order 1 or below."""
    g = torch.Generator().manual_seed(0)
    A = torch.rand(2, 3, 8, 8, generator=g, dtype=torch.float64) * 1.5 + 0.5
    b = torch.randn(2, 3, 8, 8, generator=g, dtype=torch.float64) * 0.5
    x = torch.randn(2, 3, 8, 8, generator=g, dtype=torch.float64)

    def model(v):
        return torch.tanh(A * v + b)

    r0 = 0.9
    ref = dpmpp_2m_sample_loop(model, x, logsnr_grid(2560, r0), 0.0)

    def err(n, order):
        return (dpmpp_2m_sample_loop(model, x, logsnr_grid(n, r0), 0.0, order=order) - ref).abs().max().item()

    p2 = math.log2(err(40, 2) / err(80, 2))
    p1 = math.log2(err(40, 1) / err(80, 1))
    print(f"empirical order: 2M {p2:.3f}, first order {p1:.3f}")
    assert p2 >= 1.8
    assert 0.8 <= p1 <= 1.2


def test_oracle_eta1_first_order_is_the_ancestral_update():
    """With c = 0 (order=1) the oracle's step at eta 1 is oracle.posterior_step's DDPM ancestral step."""
    from oracle.sampler import posterior_step
    g = torch.Generator().manual_seed(1)
    x = torch.randn(1, 3, 4, 4, generator=g, dtype=torch.float64)
    z = torch.randn(3, 1, 3, 4, 4, generator=g, dtype=torch.float64)
    grid = [1.0, 0.5, 0.1, 0.0]

    def model(v):
        return 0.5 * torch.tanh(v)

    want = x
    for i in range(3):
        want = posterior_step(want, model(want), grid[i], grid[i + 1], z[i], 1.0)
    got = dpmpp_2m_sample_loop(model, x, grid, 1.0, noises=z, order=1)
    assert torch.allclose(got, want, rtol=0, atol=1e-13)


# ---- ABI and CLI --------------------------------------------------------------------------------------------------
def test_op_size_and_posterior_2m_fields():
    assert ctypes.sizeof(_lib.Op) == 480
    P = _lib.Posterior2mParams
    assert ctypes.sizeof(P) == 128
    assert (P.base.offset, P.x0_prev.offset, P.c.offset) == (0, 112, 120)
    assert _lib.OP_POSTERIOR_2M == 33
    lib = _lib.load()
    assert lib.d3fk_sizeof_op() == 480
    assert hasattr(lib, "d3fk_posterior_2m_step") and "d3fk_posterior_2m_step" in _lib.EXPORTS


def test_cli_sample_lists_solver_and_schedule():
    from click.testing import CliRunner
    from denoising_diffusion_deep_fake_b200.main import cli
    res = CliRunner().invoke(cli, ["sample", "--help"])
    assert res.exit_code == 0
    assert "--solver" in res.output and "dpmpp-2m" in res.output
    assert "--schedule" in res.output and "logsnr" in res.output
    for bad in (["--solver", "dpmpp_3m"], ["--schedule", "cosine"]):
        res = CliRunner().invoke(cli, ["sample"] + bad)
        assert res.exit_code == 2 and "Invalid value" in res.output
