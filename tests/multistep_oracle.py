"""Float64 definition of the second-order multistep sampler (DPM-Solver++ 2M in data-prediction form, written in the
variance-preserving ratio r), independent of the package.  TEST INFRASTRUCTURE ONLY.

lambda(r) = ln((1 - r)/r)/2, alpha = sqrt(1 - r), s = sqrt(r).  Step i goes from r_i = grid[i] to r_t = grid[i + 1],
h_i = lambda(r_t) - lambda(r_i):
    D_i     = x0_i + c_i*(x0_i - x0_{i-1}),   c_i = h_i/(2 h_{i-1})   (0 on the first step and where h_i or h_{i-1} is
                                                                       infinite)
    x_{i+1} = (s_t/s_i) e^{-eta h} x_i + alpha_t (1 - e^{-(1+eta) h}) D_i + s_t sqrt(1 - e^{-2 eta h}) z
A step to r_t = 0 (or from r_i = 0) returns x0_i.  Masked: the blend of tests/masked_oracle.py,
x_{i+1} = m*x_{i+1} + (1 - m)*(sqrt(1 - r_t) src + sqrt(r_t) n), src itself at r_t = 0."""
import math

import torch


def lam(r):
    r = float(r)
    if r >= 1.0:
        return -math.inf
    if r <= 0.0:
        return math.inf
    return 0.5 * math.log((1.0 - r) / r)


def logsnr_grid(n_steps, r_start=1.0, r_min=1e-3):
    """n_steps + 1 ratios: r_start, then points uniform in lambda down to r_min, then 0 ([r_start, 0] for one step)."""
    if n_steps == 1:
        return [float(r_start), 0.0]
    la, lb = lam(min(r_start, 1.0 - r_min)), lam(r_min)
    grid = [1.0 / (1.0 + math.exp(2.0 * (la + (lb - la) * k / (n_steps - 1)))) for k in range(n_steps)] + [0.0]
    grid[0] = float(r_start)
    return grid


def _step(x, D, r_i, r_t, eta, z):
    """One step of the update above from r_i to r_t > 0 with the extrapolated D."""
    h = lam(r_t) - lam(r_i)
    a_t, s_t = math.sqrt(1.0 - r_t), math.sqrt(r_t)
    if math.isinf(h):                       # from pure noise: s_i = 1, e^{-k h} = 0 for k > 0, e^0 = 1
        decay = 1.0 if eta == 0.0 else 0.0
        out = s_t * decay * x + a_t * D
        sigma = s_t if eta > 0.0 else 0.0
    else:
        out = (s_t / math.sqrt(r_i)) * math.exp(-eta * h) * x + a_t * (1.0 - math.exp(-(1.0 + eta) * h)) * D
        sigma = s_t * math.sqrt(1.0 - math.exp(-2.0 * eta * h))
    if sigma > 0.0:
        if z is None:
            raise ValueError("eta > 0 needs the step's noise")
        out = out + sigma * z
    return out


@torch.no_grad()
def dpmpp_2m_sample_loop(model, x_start, grid, eta, noises=None, src=None, mask=None, known_noises=None,
                         return_trajectory=False, order=2):
    """The sampler over `grid` from x_start.  noises[i] / known_noises[i]: z and n of the step from grid index i.
    order=1 keeps c = 0 everywhere (the first-order update on the same grid)."""
    x = x_start
    x0_prev, h_prev = None, math.nan
    traj = []
    for i in range(len(grid) - 1):
        r_i, r_t = float(grid[i]), float(grid[i + 1])
        x0 = model(x)
        if r_t <= 0.0 or r_i <= 0.0:
            post, h = x0, math.nan
        else:
            h = lam(r_t) - lam(r_i)
            D = x0
            if order == 2 and x0_prev is not None and math.isfinite(h) and math.isfinite(h_prev):
                D = x0 + (h / (2.0 * h_prev)) * (x0 - x0_prev)
            post = _step(x, D, r_i, r_t, eta, None if noises is None else noises[i])
        if mask is not None:
            m = mask.clamp(0.0, 1.0)
            known = src if r_t <= 0.0 else math.sqrt(1.0 - r_t) * src + math.sqrt(r_t) * known_noises[i]
            post = m * post + (1.0 - m) * known
        x = post
        x0_prev, h_prev = x0, h
        if return_trajectory:
            traj.append(x.clone())
    return (x, traj) if return_trajectory else x
