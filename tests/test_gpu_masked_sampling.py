"""Masked (replacement-inpainting) sampling on the GPU: the masked posterior kernel against its float64 formula and its
exact contracts, its in-kernel known-region noise stream against the CPU Philox reference, the Sampler's masked mode, a
trained-weights trajectory against tests/masked_oracle.py, and the public entry points (swap_face, predict_fake, CLI).

Per-element bound of the kernel (immediate form), in units of U = 2^-24 times the magnitude of the terms each rounding
acts on — see the constants below.  The reference takes the kernel's float32 coefficients and ratio as exact."""
import copy
import math

import numpy as np
import pytest
import torch

import denoising_diffusion_deep_fake_b200 as d3
from denoising_diffusion_deep_fake_b200 import _lib
from denoising_diffusion_deep_fake_b200.functional import posterior_coeffs, posterior_step_, q_sample
from denoising_diffusion_deep_fake_b200.sampler import Sampler, swap_face
from masked_oracle import masked_sample_loop
from test_gpu_noise_streams import (LOGF_ABS, LOGF_ULP, M64, SINCOSF_ABS, SLACK, first_bad, max_ratio, normals, philox,
                                    u32_to_uniform)
from test_gpu_parity_configs import faces, oracle64, product, psnr, state_at, trained  # noqa: F401 (trained: fixture)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24
# post = fma(k_xi, x, k_x0*h), then fma(sigma, z, post): three roundings, each at most U times the sum of the term
# magnitudes T_post = |k_xi x| + |k_x0 h| + |sigma z|.
C_POST = 3
# known = fma(a, src, s*n), a = sqrtf(1 - r) (the subtraction's rounding halved by the root, plus the root's: 1.5),
# s = sqrtf(r) (1), the product (1), the fma (1): 4.5 units of T_known = |a src| + |s n|; rounded up.
C_KNOWN = 5
# out = fma(m, post, (1 - m)*known): 1 - m, the product and the fma, each at most U (|m post| + |(1 - m) known|).
C_COMP = 3


def soft_mask(B, H, W, seed):
    """[B,1,H,W] with whole 4-pixel vectors of 0 (left quarter) and of 1 (right quarter), and per-pixel values in between
    that include exact 0s and 1s and values outside [0, 1] (the kernel clamps)."""
    g = torch.Generator().manual_seed(seed)
    u = torch.rand(B, 1, H, W, generator=g) * 1.6 - 0.3
    u[..., : W // 4] = 0.0
    u[..., W - W // 4:] = 1.0
    u[..., W // 4: W // 4 + 4 * (W // 16)] = torch.where(u[..., W // 4: W // 4 + 4 * (W // 16)] > 0.5, 1.0, 0.0)
    return u.to(DEV)


def ellipse_mask(B, H, W):
    """A feathered face-like region: 1 inside an ellipse, 0 outside, a linear ramp across its edge."""
    yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float64), torch.arange(W, dtype=torch.float64), indexing="ij")
    d = torch.sqrt(((xx - (W - 1) / 2) / (0.32 * W)) ** 2 + ((yy - (H - 1) / 2) / (0.4 * H)) ** 2)
    return ((1.0 - d) / 0.15).clamp(0, 1).float().expand(B, 1, H, W).contiguous().to(DEV)


def chan(m):
    return m.expand(-1, 3, -1, -1)


# ---------------------------------------------------------------------------------------------- 1. kernel, immediate form
KERNEL_SHAPES = [(1, 128, 128), (3, 128, 128), (64, 128, 128), (256, 64, 64)]


@pytest.mark.parametrize("eta", [0.0, 1.0])
@pytest.mark.parametrize("r_i,r_prev", [(0.6, 0.4), (0.2, 0.0)])
@pytest.mark.parametrize("B,H,W", KERNEL_SHAPES)
def test_masked_posterior_kernel(B, H, W, r_i, r_prev, eta):
    g = torch.Generator().manual_seed(B + H)
    x, h, src, z, n = (torch.randn(B, 3, H, W, generator=g).to(DEV) for _ in range(5))
    m = soft_mask(B, H, W, seed=B)
    out = x.clone()
    posterior_step_(out, h, r_i, r_prev, z=z, eta=eta, src=src, mask=m, known_noise=n)
    torch.cuda.synchronize()
    # float64 formula from the kernel's float32 coefficients
    k_xi, k_x0, sigma = (float(np.float32(v)) for v in posterior_coeffs(r_i, r_prev, eta))
    r32 = float(np.float32(r_prev))
    a, s = math.sqrt(1.0 - r32), math.sqrt(r32)
    d = [t.double() for t in (x, h, src, z, n)]
    xd, hd, sd, zd, nd = d
    mc = chan(m.double().clamp(0, 1))
    post = k_xi * xd + k_x0 * hd + sigma * zd
    known = a * sd + s * nd
    ref = mc * post + (1 - mc) * known
    t_post = (k_xi * xd).abs() + (k_x0 * hd).abs() + (sigma * zd).abs()
    t_known = (a * sd).abs() + (s * nd).abs()
    bound = U * (C_POST * mc * t_post + C_KNOWN * (1 - mc) * t_known
                 + C_COMP * ((mc * post).abs() + ((1 - mc) * known).abs())) + 1e-30
    got = out.cpu().numpy().reshape(-1)
    msg = first_bad(got, ref.cpu().numpy().reshape(-1), bound.cpu().numpy().reshape(-1), "masked posterior")
    print(f"B={B} {H}x{W} r_prev {r_prev} eta {eta}: max err/bound "
          f"{max_ratio(got, ref.cpu().numpy().reshape(-1), bound.cpu().numpy().reshape(-1)):.3g}")
    assert msg is None, msg
    keep, gen = chan(m.clamp(0, 1) == 0), chan(m.clamp(0, 1) == 1)
    assert keep.any() and gen.any() and not (keep | gen).all()
    qs = q_sample(src, 1.0, noise=n, fixed_r=r_prev)
    assert torch.equal(out[keep], qs[keep])
    plain = posterior_step_(x.clone(), h, r_i, r_prev, z=z, eta=eta)
    assert torch.equal(out[gen], plain[gen])
    if r_prev == 0.0:
        assert torch.equal(out[keep], src[keep])


def test_masked_posterior_argument_checks():
    x = torch.zeros(2, 3, 8, 8, device=DEV)
    m = torch.ones(8, 8, device=DEV)
    with pytest.raises(ValueError):
        posterior_step_(x, x.clone(), 0.6, 0.4, mask=m)                                   # no src
    with pytest.raises(ValueError):
        posterior_step_(x, x.clone(), 0.6, 0.4, src=x.clone())                            # src without a mask
    with pytest.raises(ValueError):
        posterior_step_(x, x.clone(), 0.6, 0.4, src=x.clone(), mask=torch.ones(2, 3, 8, 8, device=DEV))
    with pytest.raises(ValueError):
        posterior_step_(x, x.clone(), 0.6, 0.4, src=x.clone(), mask=m.cpu())              # wrong device
    with pytest.raises(TypeError):
        posterior_step_(x, x.clone(), 0.6, 0.4, src=x.clone(), mask=m.double())
    with pytest.raises(TypeError):
        posterior_step_(x, x.clone(), 0.6, 0.4, src=x.clone().double(), mask=m)
    with pytest.raises(ValueError):
        posterior_step_(x, x.clone(), 0.6, 0.4, src=x[:1].clone(), mask=m)
    out = posterior_step_(x, x.clone(), 0.6, 0.4, src=x.clone(), mask=m.bool())         # bool [H,W] is accepted
    assert torch.equal(out, torch.zeros_like(out))


# ---------------------------------------------------------------------------------------------- 2. known-noise stream
def known_normals(seed, offset, n):
    """(float64 normals, bound) of philox_normal4(seed, i | 1 << 63, offset): normals() with bit 31 of counter word 1."""
    i = np.arange(n // 4, dtype=np.uint64)
    w = philox(i & np.uint64(M64), (i >> np.uint64(32)) | np.uint64(0x80000000), np.full_like(i, offset & M64),
               np.full_like(i, offset >> 32), seed & M64, seed >> 32)
    u = [u32_to_uniform(v) for v in w]
    out, bound = np.empty((n // 4, 4)), np.empty((n // 4, 4))
    for j, (ur, ut) in enumerate(((u[0], u[1]), (u[2], u[3]))):
        L = np.log(ur.astype(np.float64))
        dL = np.where(ur >= np.float32(0.5), LOGF_ABS, LOGF_ULP * 2.0 ** -23 * np.abs(L))
        R, dR = -2.0 * L, 2.0 * dL
        r = np.sqrt(R)
        with np.errstate(divide="ignore"):
            dr = np.minimum(np.sqrt(dR), dR / (2.0 * r)) + U * r
        t = (np.float32(6.283185307179586) * ut).astype(np.float64)
        for k, f in enumerate((np.cos, np.sin)):
            v = r * f(t)
            out[:, 2 * j + k] = v
            bound[:, 2 * j + k] = SLACK * (dr + (r + dr) * SINCOSF_ABS + U * np.abs(v))
    return out.reshape(-1), bound.reshape(-1)


def check_scaled_noise(got, s, ref, bound, what):
    msg = first_bad(got, s * ref, s * bound + U * np.abs(s * ref), what)
    assert msg is None, msg


@pytest.mark.parametrize("seed,offset", [(0, 0), (2 ** 32 + 5, 7), (2 ** 64 - 1, 2 ** 32 + 3)])
def test_known_noise_stream_immediate(seed, offset):
    """x = x0_hat = src = 0, m = 0: the output is sqrt(r_prev) * n, n from the known-region stream."""
    shape = (4, 3, 64, 96)
    zeros = torch.zeros(shape, device=DEV)
    out = zeros.clone()
    r_prev = 0.4
    posterior_step_(out, zeros, 0.6, r_prev, eta=1.0, seed=seed, offset=offset, src=zeros,
                    mask=torch.zeros(64, 96, device=DEV))
    got = out.cpu().numpy().reshape(-1)
    s = float(np.sqrt(np.float32(r_prev)))
    ref, bound = known_normals(seed, offset, got.size)
    check_scaled_noise(got, s, ref, bound, "sqrt(r_prev) * n")
    # n is none of the existing draws: not z / q_sample's noise of the same key and offset, not the sampler's start noise
    for other, _ in (normals(seed, offset, got.size), normals(seed ^ 0x5EED, 0, got.size),
                     normals(seed ^ 0x5EED, offset, got.size)):
        assert (np.abs(got - s * other) > s * bound).mean() > 0.99
    z = zeros.clone()
    posterior_step_(z, zeros, 0.6, r_prev, eta=1.0, seed=seed, offset=offset)         # sigma * z, in-kernel
    qn = q_sample(zeros, 1.0, seed=seed, offset=offset, fixed_r=1.0)                   # q_sample's noise
    for other in (z.cpu().numpy().reshape(-1) / float(np.float32(posterior_coeffs(0.6, r_prev, 1.0)[2])),
                  qn.cpu().numpy().reshape(-1)):
        assert (np.abs(got - s * other) > s * bound).mean() > 0.99


def test_known_noise_stream_graph_form():
    """The form a masked Sampler captures: coef_table[*step] = (k_xi, k_x0, sigma, r_prev), the known noise at offset +
    *step, one op pair per chain with seed + 0x9E3779B1 * c, replayed as one CUDA graph."""
    _lib.init(0)
    k_steps, chains, seed, offset = 4, 2, 2 ** 32 + 5, 7
    B, H, W = 2, 32, 64
    shape = (B, 3, H, W)
    ratios = [0.8 - 0.15 * k for k in range(k_steps)]
    coef = torch.tensor([(0.0, 0.0, 0.0, r) for r in ratios], dtype=torch.float32, device=DEV)
    xs = [torch.full(shape, 9.0, device=DEV) for _ in range(chains)]
    hs = [torch.full(shape, 9.0, device=DEV) for _ in range(chains)]
    src = torch.zeros(shape, device=DEV)
    mask = torch.zeros(B, 1, H, W, device=DEV)
    steps = [torch.zeros(1, dtype=torch.int32, device=DEV) for _ in range(chains)]
    ops = []
    for c in range(chains):
        ops.append(_lib.make_op(_lib.OP_POSTERIOR, n=xs[c].numel(), x=xs[c].data_ptr(), x0_hat=hs[c].data_ptr(),
                                coef_table=coef.data_ptr(), step=steps[c].data_ptr(), seed=seed + 0x9E3779B1 * c,
                                offset=offset, src=src.data_ptr(), mask=mask.data_ptr(), chw=3 * H * W, hw=H * W))
        ops.append(_lib.make_op(_lib.OP_INC, p0=steps[c].data_ptr(), n=1))
    ops = _lib.OpList(ops)
    stream = torch.cuda.Stream(DEV)
    stream.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(stream):
        ops.run(stream.cuda_stream)
        for st in steps:
            st.zero_()
    torch.cuda.current_stream(DEV).wait_stream(stream)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=stream):
        ops.run(stream.cuda_stream)
    for k in range(k_steps):
        graph.replay()
        torch.cuda.synchronize()
        s = float(np.sqrt(np.float32(ratios[k])))
        for c in range(chains):
            assert steps[c].item() == k + 1
            got = xs[c].cpu().numpy().reshape(-1)
            ref, bound = known_normals(seed + 0x9E3779B1 * c, offset + k, got.size)
            check_scaled_noise(got, s, ref, bound, f"chain {c} step {k}")
    assert _lib.load().d3fk_device_error_flag() == 0


# ---------------------------------------------------------------------------------------------- 3. Sampler contracts
@pytest.fixture(scope="module")
def small_model():
    torch.manual_seed(0)
    return d3.Unet(precision="bf16").to(DEV).eval()


def _src(B, H, W, seed=11):
    return faces(B, H, W, seed)


@pytest.mark.parametrize("eta", [0.0, 1.0])
@pytest.mark.parametrize("chains", [1, 2])
def test_sampler_mask_of_ones_is_unmasked(small_model, eta, chains):
    B, H, W, n = 4, 64, 64, 5
    plain = Sampler(small_model, B, H, W, n, eta=eta, seed=3, chains=chains).run()
    smp = Sampler(small_model, B, H, W, n, eta=eta, seed=3, chains=chains, masked=True)
    assert smp.kernels_per_step == Sampler(small_model, B, H, W, n, eta=eta, seed=3, chains=chains).kernels_per_step
    out = smp.run(src=_src(B, H, W), mask=torch.ones(H, W, device=DEV))
    assert torch.equal(out, plain)
    assert _lib.load().d3fk_device_error_flag() == 0


def test_sampler_mask_of_zeros_returns_src(small_model):
    B, H, W = 4, 64, 64
    src = _src(B, H, W)
    out = Sampler(small_model, B, H, W, 6, r_start=0.6, eta=1.0, seed=5, masked=True).run(
        src=src, mask=torch.zeros(1, 1, H, W, device=DEV))
    assert torch.equal(out, src)


def test_sampler_masked_replay_eager_and_launches(small_model):
    B, H, W, n = 4, 64, 64, 6
    src, m = _src(B, H, W), ellipse_mask(B, H, W)
    smp = Sampler(small_model, B, H, W, n, r_start=0.7, eta=0.0, seed=9, masked=True)
    a = smp.run(src=src, mask=m)
    b = smp.run(src=src, mask=m)
    assert torch.equal(a, b)                                               # graph replay is repeatable
    assert torch.equal(a[chan(m == 0)], src[chan(m == 0)])
    # eager path (noises given, known_noises=None) draws the graph's known noise: seed, offset = step
    eager = smp.run(src=src, mask=m, noises=torch.zeros(n, B, 3, H, W, device=DEV))
    assert torch.equal(eager, a)
    # the mask adds no launch
    counts = []
    for masked in (False, True):
        s = Sampler(small_model, B, H, W, n, r_start=0.7, seed=9, use_graph=False, masked=masked)
        kw = dict(src=src, mask=m) if masked else {}
        s.run(**kw)
        before = _lib.launch_count()
        s.run(**kw)
        counts.append(_lib.launch_count() - before)
    assert counts[0] == counts[1]
    with pytest.raises(ValueError):
        smp.run()                                                          # a masked sampler needs src and mask
    assert _lib.load().d3fk_device_error_flag() == 0


# ---------------------------------------------------------------------------------------------- 4. trajectory parity
@pytest.mark.parametrize("precision,B,H,eta", [("bf16", 4, 64, 0.0), ("bf16", 64, 128, 0.0), ("bf16", 16, 128, 1.0),
                                              ("fp32", 4, 64, 0.0)])
def test_masked_trajectory_psnr_benchmarked_configs(trained, precision, B, H, eta):  # noqa: F811
    """20-step masked trajectories with supplied noises and known noises against masked_sample_loop in float64, at the
    thresholds of test_gpu_parity_configs.py::test_sampler_trajectory_psnr_benchmarked_configs; the known region is the
    source exactly at the end."""
    ref = trained[0]
    sd = state_at(trained, H)
    n_steps = 20
    g = torch.Generator(device=DEV).manual_seed(5)
    x_start = torch.randn(B, 3, H, H, generator=g, device=DEV)
    noises = torch.randn(n_steps, B, 3, H, H, generator=g, device=DEV) if eta > 0 else None
    known = torch.randn(n_steps, B, 3, H, H, generator=g, device=DEV)
    src = faces(B, H, H, seed=17)
    m = ellipse_mask(B, H, H)
    r64 = oracle64(ref, sd, False)
    out64 = masked_sample_loop(r64, x_start.double(), src.double(), m.double(), n_steps, eta=eta,
                               noises=None if noises is None else noises.double(), known_noises=known.double())
    model = product(precision, sd, False)
    out = Sampler(model, B, H, H, n_steps, eta=eta, masked=True).run(x_start, noises=noises, src=src, mask=m,
                                                                     known_noises=known)
    p = psnr(out, out64)
    p_lib = None
    if precision == "bf16":
        lib = copy.deepcopy(ref)
        lib.load_state_dict(sd)
        lib = lib.to(DEV).eval().to(memory_format=torch.channels_last)

        def lib_model(x):
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                return lib(x.float().contiguous(memory_format=torch.channels_last)).float()

        out_lib = masked_sample_loop(lib_model, x_start, src, m, n_steps, eta=eta, noises=noises, known_noises=known)
        p_lib = psnr(out_lib, out64)
        del lib
    print(f"masked final PSNR {p:.2f} dB" + (f" | torch bf16 autocast {p_lib:.2f} dB" if p_lib is not None else ""))
    assert p >= 40.0 or (p_lib is not None and p >= p_lib - 0.5), (precision, B, H, eta, p, p_lib)
    keep = chan(m == 0)
    assert torch.equal(out[keep], src[keep])
    assert d3._lib.load().d3fk_device_error_flag() == 0


# ---------------------------------------------------------------------------------------------- 5. public entry points
def test_swap_face_mask(small_model):
    B, H, W = 3, 64, 64
    real = _src(B, H, W, seed=21)
    m = soft_mask(B, H, W, seed=4)
    with torch.no_grad():
        fake = small_model(real)
    out = swap_face(small_model, real, mask=m)
    mc = chan(m.clamp(0, 1))
    assert torch.equal(out[mc == 0], real[mc == 0]) and torch.equal(out[mc == 1], fake[mc == 1])
    ref = mc.double() * fake.double() + (1 - mc.double()) * real.double()
    assert torch.allclose(out.double(), ref, rtol=0, atol=1e-5)
    assert torch.equal(swap_face(small_model, real), fake)                 # mask=None: unchanged
    m2 = m[0, 0].cpu()                                                     # an [H,W] mask on the host, for every sample
    out2 = swap_face(small_model, real, n_steps=4, r_start=0.5, eta=1.0, seed=2, mask=m2)
    keep2 = (m2.clamp(0, 1) == 0).to(DEV).expand(B, 3, H, W)
    assert torch.isfinite(out2).all() and torch.equal(out2[keep2], real[keep2])


@pytest.fixture(scope="module")
def deep_fake_module():
    from denoising_diffusion_deep_fake_b200.train import DeepFakeModule
    torch.manual_seed(0)
    return DeepFakeModule(encoder_name="resnet34", learning_rate=1e-3, noise_exponential_sampling_lambda=3, mode="denoise",
                          mean_a=[0.5, 0.5, 0.5], std_a=[0.5, 0.5, 0.5], mean_b=[0.45, 0.5, 0.55],
                          std_b=[0.4, 0.5, 0.6], precision="fp32").to(DEV)


def test_predict_fake_mask_on_frames(deep_fake_module):
    from denoising_diffusion_deep_fake_b200.functional import frames_to_tensor, tensor_to_frames
    mod = deep_fake_module
    mean, std = [0.45, 0.5, 0.55], [0.4, 0.5, 0.6]                        # model "a" uses mean_b / std_b
    rng = np.random.default_rng(5)
    frame = rng.integers(0, 256, size=(64, 64, 3), dtype=np.uint8)
    mask = np.zeros((64, 64), np.uint8)
    mask[16:48, 20:44] = 255
    mask[16:48, 18:20] = 128                                               # a feathered edge
    fake = mod.predict_fake(frame, "a", mask=mask)
    plain = mod.predict_fake(frame, "a")
    assert isinstance(fake, np.ndarray) and fake.dtype == np.uint8 and fake.shape == frame.shape
    round_trip = tensor_to_frames(frames_to_tensor(torch.from_numpy(frame).to(DEV), mean, std), mean, std)[0].cpu().numpy()
    assert np.array_equal(fake[mask == 0], round_trip[mask == 0])
    assert np.array_equal(fake[mask == 255], plain[mask == 255])
    # mask=None is unchanged: the network's frame
    x = frames_to_tensor(torch.from_numpy(frame).to(DEV), mean, std)
    with torch.no_grad():
        mod.model_a.eval()
        want = tensor_to_frames(mod.model_a(x), mean, std)[0].cpu().numpy()
    assert np.array_equal(plain, want)
    # a CUDA batch with an [N,H,W] uint8 mask
    batch = torch.from_numpy(np.stack([frame, frame[::-1].copy()])).to(DEV)
    masks = torch.from_numpy(np.stack([mask, mask[:, ::-1].copy()])).to(DEV)
    out = mod.predict_fake(batch, "a", mask=masks)
    assert out.is_cuda and np.array_equal(out[0].cpu().numpy(), fake)
    rt = tensor_to_frames(frames_to_tensor(batch, mean, std), mean, std)
    keep = (masks == 0).unsqueeze(-1).expand_as(rt)
    assert torch.equal(out[keep], rt[keep])


def test_predict_fake_mask_on_tensors(deep_fake_module):
    mod = deep_fake_module
    real = _src(2, 64, 64, seed=8)
    m = soft_mask(2, 64, 64, seed=6)
    out = mod.predict_fake(real, "b", mask=m)
    fake = mod.predict_fake(real, "b")
    mc = chan(m.clamp(0, 1))
    assert torch.equal(out[mc == 0], real[mc == 0]) and torch.equal(out[mc == 1], fake[mc == 1])
    with pytest.raises(TypeError):
        mod.predict_fake(real, "b", mask=(m > 0.5).to(torch.uint8))     # uint8 masks are for uint8 frames


def test_cli_sample_source_mask(tmp_path):
    from click.testing import CliRunner
    from denoising_diffusion_deep_fake_b200.main import cli
    B, H, W = 2, 64, 96
    src = faces(B, H, W, seed=3).cpu()
    m = torch.zeros(H, W)
    m[16:48, 24:72] = 1.0
    torch.save(src, tmp_path / "src.pt")
    torch.save(m, tmp_path / "mask.pt")
    res = CliRunner().invoke(cli, ["sample", "--source", str(tmp_path / "src.pt"), "--mask", str(tmp_path / "mask.pt"),
                                   "--steps", "4", "--r_start", "0.6", "--eta", "1.0", "--out", str(tmp_path / "o.pt")])
    assert res.exit_code == 0, res.output
    out = torch.load(tmp_path / "o.pt")
    keep = (m == 0).expand(B, 3, H, W)
    assert out.shape == src.shape and torch.equal(out[keep], src[keep])
    assert torch.isfinite(out).all()
