"""Float64 definition of masked (replacement-inpainting) sampling on top of oracle.sampler, which it leaves as it is.
TEST INFRASTRUCTURE ONLY.

Step i goes from ratio r_i to r_prev = r_{i+1}:
    post    = k_xi * x_i + k_x0 * x0_hat + sigma * z          (oracle.posterior_step)
    known   = sqrt(1 - r_prev) * src + sqrt(r_prev) * n        (src at r_prev = 0)
    x_{i+1} = m * post + (1 - m) * known                       (m = mask clamped to [0, 1], broadcast over channels)
so the last step gives m * x0_hat + (1 - m) * src, and n_steps = 1, r_start = 0 is m * model(src) + (1 - m) * src."""
import math

import torch

from oracle.sampler import noise_ratio_grid, posterior_step


def masked_posterior_step(x_i, x0_hat, r_i, r_prev, src, mask, z=None, n=None, eta=0.0):
    post = posterior_step(x_i, x0_hat, r_i, r_prev, z, eta)
    r_prev = float(r_prev)
    known = src if r_prev <= 0.0 else math.sqrt(1.0 - r_prev) * src + math.sqrt(r_prev) * n
    m = mask.clamp(0.0, 1.0)
    return m * post + (1.0 - m) * known


@torch.no_grad()
def masked_sample_loop(model, x_start, src, mask, n_steps, r_start=1.0, eta=0.0, noises=None, known_noises=None,
                       return_trajectory=False):
    """oracle.sample_loop with the known region replaced at every step; known_noises[i] is n of the step from grid
    index i (unused where r_prev = 0)."""
    grid = noise_ratio_grid(n_steps, r_start).tolist()
    x = x_start
    traj = []
    for i in range(n_steps):
        x0_hat = model(x)
        z = None if noises is None else noises[i]
        n = None if known_noises is None else known_noises[i]
        x = masked_posterior_step(x, x0_hat, grid[i], grid[i + 1], src, mask, z, n, eta)
        if return_trajectory:
            traj.append(x.clone())
    return (x, traj) if return_trajectory else x
