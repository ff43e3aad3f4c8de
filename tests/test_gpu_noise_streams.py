"""The in-kernel Philox noise streams of q_sample and the posterior step against a reference reproduced on the CPU.

Reference.  Philox4x32-10 is integer arithmetic: `philox` below (numpy, 64-bit products) reproduces it exactly and is
checked against the Random123 known-answer vectors.  Uniforms are reproduced bit for bit in numpy float32 as
u32_to_uniform forms them (common.cuh): round-to-nearest (float)u, + 0.5f, * 2^-32.  The add and the multiply cannot contract
into one FMA, and the library is built without fast-math.  From those uniforms the normals are Box-Muller in float64 in the
element order of philox_normal4: counter (i, i >> 32, offset, offset >> 32) for the 4-element vector i, key
(seed, seed >> 32), elements (ra cos t1, ra sin t1, rb cos t3, rb sin t3) with ra = sqrt(-2 log u0), rb = sqrt(-2 log u2)
and the angle t = (float)(2 pi) * u rounded to float32 as the kernel rounds it.  The per-sample ratio of q_sample is the
draw with counter (b, 0, offset, 0x9E3779B9): y = (x >> 8) * 2^-24, r = clamp(1/lam * log(1 / (y (1 - e^-lam) + e^-lam)), 0, 1).

Bounds, per element, derived in the table below.  Any error in a counter, key or offset changes essentially every element
by O(1), so a bound generous by a small factor costs no sensitivity (test_bounds_separate_wrong_streams shows that each
such slip moves nearly every element past its bound).

affine_q_sample draws its noise and ratio with the same counters and its fused output equals q_sample of the warped image
bit for bit (test_gpu_elementwise.py::test_affine_q_sample), so it needs no reference of its own here."""
import math

import numpy as np
import pytest
import torch

import denoising_diffusion_deep_fake_b200 as d3
from denoising_diffusion_deep_fake_b200 import _lib

DEV = "cuda:0"
M64 = 0xFFFFFFFF

# ---- constants ----
U = 2.0 ** -24                   # fp32 unit roundoff
LOGF_ABS = 2.0 ** -21.41         # __logf on [0.5, 2]: maximum absolute error (CUDA programming guide, intrinsic functions)
# __logf below 0.5: the guide gives 3 ulp; measured exhaustively over the uniforms in [2^-33, 0.5) on an NVIDIA B200
# (tools/probes/fastmath_error.cu), the maximum is 3.34 ulp, so the bound takes 4.  (On [0.5, 1] it measured 2^-22.45.)
LOGF_ULP = 4
# __sincosf: the guide documents 2^-21.41 absolute on [-pi, pi] only; the kernel's angle reaches 2 pi.  Maximum absolute
# error of sin and cos over every float32 angle in [0, (float)(2 pi)], measured exhaustively on an NVIDIA B200 with the same
# probe: 2^-20.55 (sin) and 2^-20.43 (cos), rounded up to the next quarter power of two.
SINCOSF_ABS = 2.0 ** -20.25
SLACK = 2.0                      # the normal bound is doubled: first-order terms only, and it costs no sensitivity (above)
# Ratio draw: expf(-lam) (2 ulp = 4U relative), 1 - c, the multiply-add and the division (1U each) give the argument of
# logf a relative error of 7U, i.e. an absolute error of 7U in its log; logf adds 1 ulp (2U relative) and 1/lam and the
# final product 1U each: |dr| <= U * (T_R_ABS / lam + T_R_REL * r), with one unit of slack in each.
T_R_ABS = 8
T_R_REL = 5

SEEDS = [0, 123, 2 ** 32 + 5, 2 ** 64 - 1]
OFFSETS = [0, 7, 2 ** 32 + 3]


# ---------------------------------------------------------------------------------------------------------------------
# reference

def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on uint64 arrays holding 32-bit words (the products need the full 64 bits)."""
    c = [np.asarray(v, dtype=np.uint64) for v in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    m, s = np.uint64(M64), np.uint64(32)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> s) ^ c[1] ^ k0, p1 & m, (p0 >> s) ^ c[3] ^ k1, p0 & m]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m, (k1 + np.uint64(0xBB67AE85)) & m
    return c


def u32_to_uniform(u):
    return (np.asarray(u).astype(np.uint32).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -32)


def normals(seed, offset, n):
    """(float64 normals, float64 per-element bound) of the first n elements of philox_normal4(seed, i, offset)."""
    i = np.arange(n // 4, dtype=np.uint64)
    w = philox(i & np.uint64(M64), i >> np.uint64(32), np.full_like(i, offset & M64), np.full_like(i, offset >> 32),
               seed & M64, seed >> 32)
    u = [u32_to_uniform(v) for v in w]
    out, bound = np.empty((n // 4, 4)), np.empty((n // 4, 4))
    for j, (ur, ut) in enumerate(((u[0], u[1]), (u[2], u[3]))):
        L = np.log(ur.astype(np.float64))
        dL = np.where(ur >= np.float32(0.5), LOGF_ABS, LOGF_ULP * 2.0 ** -23 * np.abs(L))
        R, dR = -2.0 * L, 2.0 * dL
        r = np.sqrt(R)
        with np.errstate(divide="ignore"):
            dr = np.minimum(np.sqrt(dR), dR / (2.0 * r)) + U * r            # sqrtf rounds once
        t = (np.float32(6.283185307179586) * ut).astype(np.float64)        # the kernel's float32 angle, exactly
        for k, f in enumerate((np.cos, np.sin)):
            v = r * f(t)
            out[:, 2 * j + k] = v
            bound[:, 2 * j + k] = SLACK * (dr + (r + dr) * SINCOSF_ABS + U * np.abs(v))   # + the product's rounding
    return out.reshape(-1), bound.reshape(-1)


def ratios(B, seed, offset, lam):
    """(float64 r, bound) of q_sample's per-sample draw."""
    w = philox(np.arange(B, dtype=np.uint64), np.zeros(B, np.uint64), np.full(B, offset & M64, np.uint64),
               np.full(B, 0x9E3779B9, np.uint64), seed & M64, seed >> 32)
    y = (w[0] >> np.uint64(8)).astype(np.float64) * 2.0 ** -24
    c = math.exp(-lam)
    r = np.clip((1.0 / lam) * np.log(1.0 / (y * (1.0 - c) + c)), 0.0, 1.0)
    return r, U * (T_R_ABS / lam + T_R_REL * r)


def first_bad(got, ref, bound, what):
    err = np.abs(got.astype(np.float64) - ref)
    bad = ~(err <= bound)
    if not bad.any():
        return None
    k = int(np.flatnonzero(bad)[0])
    return (f"{what}: {int(bad.sum())} of {bad.size} elements over the bound; first at flat index {k} (vector {k // 4}, "
            f"lane {k % 4}): got {got[k]!r} ref {ref[k]!r} err {err[k]:.3e} bound {bound[k]:.3e}")


def max_ratio(got, ref, bound):
    return float((np.abs(got.astype(np.float64) - ref) / bound).max())


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests

KAT = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
       ((M64,) * 4, (M64, M64), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
       ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
        (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_philox_known_answers(ctr, key, want):
    """Random123's known-answer vectors for Philox4x32-10."""
    got = tuple(int(v[0]) for v in philox(*[np.array([x], np.uint64) for x in ctr], *key))
    assert got == want, " ".join(f"{v:08x}" for v in got)


def test_uniform_conversion():
    """u32_to_uniform: (float)u rounds to nearest even, then + 0.5f and * 2^-32 each round once; (0, 1]."""
    u = np.array([0, 1, 2 ** 24, 2 ** 24 + 1, 2 ** 24 + 3, 2 ** 31, M64 - 128, M64 - 127, M64], dtype=np.uint64)
    got = u32_to_uniform(u)
    want = np.array([2.0 ** -33, 1.5 * 2.0 ** -32, 2.0 ** -8, 2.0 ** -8, (2 ** 24 + 4) * 2.0 ** -32, 0.5, 1 - 2.0 ** -24,
                     1.0, 1.0], dtype=np.float32)
    assert got.dtype == np.float32 and np.array_equal(got, want), got


def test_bounds_separate_wrong_streams():
    """Each slip a statistics test would pass (the seed's high word dropped, the offset's high word dropped, every sample
    drawing the same noise, the offset left out of the ratio draw) moves nearly every element past its bound."""
    n = 4 * 3 * 32 * 32
    ref, bound = normals(2 ** 32 + 5, 2 ** 32 + 3, n)
    for wrong in (normals(5, 2 ** 32 + 3, n)[0], normals(2 ** 32 + 5, 3, n)[0],
                  np.tile(ref[:n // 4], 4)):
        moved = np.abs(wrong - ref) > bound
        assert moved[n // 4:].mean() > 0.99
    r, rb = ratios(256, 123, 7, 5.0)
    assert (np.abs(ratios(256, 123, 0, 5.0)[0] - r) > rb).mean() > 0.99
    assert bound.max() < 1e-3 and rb.max() < 1e-6


# ---------------------------------------------------------------------------------------------------------------------
# GPU tests

def _qsample_cases():
    cases = [((256, 3, 64, 64), 123, 7), ((256, 3, 64, 64), 2 ** 64 - 1, 2 ** 32 + 3)]
    cases += [(s, seed, off) for s in [(5, 3, 128, 96), (1, 3, 32, 32)] for seed in SEEDS for off in OFFSETS]
    return [pytest.param(s, seed, off, id=f"{'x'.join(map(str, s))}-seed{seed}-off{off}") for s, seed, off in cases]


@pytest.mark.gpu
@pytest.mark.parametrize("fixed_r", [None, 0.7])
@pytest.mark.parametrize("shape,seed,offset", _qsample_cases())
def test_q_sample_streams(shape, seed, offset, fixed_r):
    """noise_out and r_out of q_sample with the in-kernel draws, and out = sqrt(1 - r) x + sqrt(r) noise from them."""
    B = shape[0]
    x = torch.rand(shape, generator=torch.Generator().manual_seed(0)) * 2 - 1
    out, noise, r = d3.q_sample(x.to(DEV), 5.0, seed=seed, offset=offset, fixed_r=fixed_r, return_aux=True)
    noise, r, out = noise.cpu().numpy().reshape(-1), r.cpu().numpy().reshape(-1), out.cpu().numpy().reshape(-1)
    ref_n, bound_n = normals(seed, offset, noise.size)
    if fixed_r is None:
        ref_r, bound_r = ratios(B, seed, offset, 5.0)
    else:
        ref_r, bound_r = np.full(B, float(np.float32(fixed_r))), np.zeros(B)
    print(f"q_sample {shape} seed {seed} offset {offset} fixed_r {fixed_r}: max err/bound noise "
          f"{max_ratio(noise, ref_n, bound_n):.3g} r {max_ratio(r, ref_r, np.maximum(bound_r, 1e-300)):.3g}")
    msg = first_bad(noise, ref_n, bound_n, "noise")
    assert msg is None, msg
    msg = first_bad(r, ref_r, bound_r, "r")
    assert msg is None, msg
    # the blend uses these very draws: kernel r and noise in, float64 blend out, rounding of sqrt, product and fma
    rr = np.repeat(r.astype(np.float64), noise.size // B)
    a, s = np.sqrt(1.0 - rr), np.sqrt(rr)
    xs = x.numpy().reshape(-1).astype(np.float64)
    msg = first_bad(out, a * xs + s * noise, 4 * U * (np.abs(a * xs) + np.abs(s * noise)) + 1e-30, "out")
    assert msg is None, msg


@pytest.mark.gpu
@pytest.mark.parametrize("seed,offset", [(0, 0), (2 ** 32 + 5, 7), (2 ** 64 - 1, 2 ** 32 + 3)])
def test_posterior_step_stream(seed, offset):
    """posterior_step_ with no z and eta > 0 draws z in-kernel; with x = x0_hat = 0 the output is sigma * z."""
    shape = (4, 3, 64, 96)
    x = torch.zeros(shape, device=DEV)
    h = torch.zeros(shape, device=DEV)
    r_i, r_prev = 0.6, 0.4
    sigma = float(np.float32(d3.functional.posterior_coeffs(r_i, r_prev, 1.0)[2]))
    assert sigma > 0
    d3.posterior_step_(x, h, r_i, r_prev, eta=1.0, seed=seed, offset=offset)
    got = x.cpu().numpy().reshape(-1)
    ref, bound = normals(seed, offset, got.size)
    msg = first_bad(got, sigma * ref, sigma * bound + U * np.abs(sigma * ref), "sigma * z")
    assert msg is None, msg


@pytest.mark.gpu
def test_sampler_graph_form_streams():
    """The form Sampler captures: OP_POSTERIOR reading its coefficients from coef_table[*step] and drawing z at offset
    + *step, then OP_INC, one pair per chain with seed + 0x9E3779B1 * c, replayed as one CUDA graph k times.  With
    k_xi = k_x0 = 0 every replay leaves sigma_k * z_k: step k must use table row k and offset + k."""
    _lib.init(0)
    k_steps, chains, seed, offset = 4, 2, 2 ** 32 + 5, 7
    shape = (2, 3, 32, 64)
    coef = torch.tensor([(0.0, 0.0, 0.5 + 0.25 * k, 0.0) for k in range(k_steps)], dtype=torch.float32, device=DEV)
    xs = [torch.full(shape, 9.0, device=DEV) for _ in range(chains)]
    hs = [torch.full(shape, 9.0, device=DEV) for _ in range(chains)]
    steps = [torch.zeros(1, dtype=torch.int32, device=DEV) for _ in range(chains)]
    ops = []
    for c in range(chains):
        ops.append(_lib.make_op(_lib.OP_POSTERIOR, n=xs[c].numel(), x=xs[c].data_ptr(), x0_hat=hs[c].data_ptr(),
                                coef_table=coef.data_ptr(), step=steps[c].data_ptr(),
                                seed=seed + 0x9E3779B1 * c, offset=offset))
        ops.append(_lib.make_op(_lib.OP_INC, p0=steps[c].data_ptr(), n=1))
    ops = _lib.OpList(ops)
    stream = torch.cuda.Stream(DEV)
    stream.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(stream):                    # warm-up launch outside capture, as Sampler does
        ops.run(stream.cuda_stream)
        for s in steps:
            s.zero_()
    torch.cuda.current_stream(DEV).wait_stream(stream)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=stream):
        ops.run(stream.cuda_stream)
    for k in range(k_steps):
        graph.replay()
        torch.cuda.synchronize()
        sigma = 0.5 + 0.25 * k
        for c in range(chains):
            assert steps[c].item() == k + 1
            got = xs[c].cpu().numpy().reshape(-1)
            ref, bound = normals(seed + 0x9E3779B1 * c, offset + k, got.size)
            msg = first_bad(got, sigma * ref, sigma * bound + U * np.abs(sigma * ref), f"chain {c} step {k}")
            assert msg is None, msg
