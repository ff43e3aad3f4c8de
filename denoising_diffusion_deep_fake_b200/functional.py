"""Fused elementwise entry points of the hot path: noising (q_sample) and the posterior update.

q_sample replaces `LitModule.blend_random_amount_of_noise_with_each_sample` +
`sample_random_number_from_exponential_distribution` (d3f/train_denoiser/lit_module.py:128-153,
duplicated at d3f/train_deep_fake/lit_module.py:208-233) — ~10 eager launches -> 1 kernel.
posterior_step is the sampler update of SURVEY §8a row S (no reference counterpart)."""
import math

import torch

from . import _lib
from ._lib import make_op


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _require_cuda_f32(t, name):
    if not t.is_cuda:
        raise _lib.D3fkError(f"{name}: d3fk kernels need a CUDA (sm_100a) tensor; there is no CPU path")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32")
    _lib.init(t.device.index)


def composite_(out, src, mask):
    """In place: out = m*out + (1 - m)*src (mask as normalize_mask accepts) — the masked posterior of the last step, whose
    known region is the source itself; exactly src where m == 0 and out where m == 1."""
    return posterior_step_(out, out, 0.0, 0.0, src=src, mask=mask)


def q_sample(batch, lam, noise=None, y=None, seed=0, offset=0, fixed_r=None, return_aux=False, out=None):
    """noisy = sqrt(1-r)*batch + sqrt(r)*noise with per-sample r = 1/lam*log(1/(y(1-c)+c)), c = e^-lam.
    noise / y: optional tensors (parity with the reference's torch.randn_like / torch.rand draws);
    otherwise drawn in-kernel from Philox4x32-10(seed, offset)."""
    _require_cuda_f32(batch, "batch")
    batch = batch.contiguous()
    B = batch.shape[0]
    if out is None:
        out = torch.empty_like(batch)
    elif out.shape != batch.shape or out.dtype != torch.float32 or not out.is_contiguous() or out.device != batch.device:
        raise ValueError("q_sample: `out` must be a contiguous float32 tensor of the batch's shape on its device")
    r_out = torch.empty(B, dtype=torch.float32, device=batch.device) if return_aux else None
    n_out = torch.empty_like(batch) if (return_aux and noise is None) else None
    if noise is not None:
        noise = noise.contiguous()
    if y is not None:
        y = y.reshape(B).contiguous()
    op = make_op(_lib.OP_QSAMPLE, B=B, chw=batch[0].numel(), lam=float(lam),
                 fixed_r=-1.0 if fixed_r is None else float(fixed_r), x=batch.data_ptr(),
                 noise=None if noise is None else noise.data_ptr(), y=None if y is None else y.data_ptr(),
                 out=out.data_ptr(), r_out=None if r_out is None else r_out.data_ptr(),
                 noise_out=None if n_out is None else n_out.data_ptr(), seed=int(seed), offset=int(offset))
    _lib.run_single(op, _stream(batch))
    if return_aux:
        return out, (noise if noise is not None else n_out), r_out.view(B, 1, 1, 1)
    return out


def noise_ratio_grid(n_steps, r_start=1.0, kind="linear", r_min=1e-3):
    """The sampler's ratios r_start = grid[0] > ... > grid[n_steps] = 0.
    kind="linear": linear in r (alpha_bar = 1 - r).
    kind="logsnr": uniform in lambda(r) = ln((1 - r)/r)/2 from lambda(min(r_start, 1 - r_min)) to lambda(r_min) over the
    first n_steps points, then 0; grid[0] is r_start itself, so from r_start = 1 the first step goes straight from pure
    noise to the second point.  n_steps = 1 is [r_start, 0].  The last nonzero ratio is r_min whatever n_steps, so the
    trajectory ends at the same point for every step count (the linear grid's ends at r_start/n_steps)."""
    if kind == "linear":
        return [r_start * (1.0 - i / n_steps) for i in range(n_steps + 1)]
    if kind != "logsnr":
        raise ValueError(f"unknown grid kind {kind!r}: 'linear' or 'logsnr'")
    if n_steps < 1:
        raise ValueError(f"n_steps must be at least 1, got {n_steps}")
    if not 0.0 < r_min < 0.5:
        raise ValueError(f"r_min must lie in (0, 0.5), got {r_min}")
    r_start = float(r_start)
    if not 0.0 <= r_start <= 1.0:
        raise ValueError(f"r_start must lie in [0, 1], got {r_start}")
    if r_start == 0.0:
        return [0.0] * (n_steps + 1)
    if n_steps == 1:
        return [r_start, 0.0]
    if r_start <= r_min:
        raise ValueError(f"a logsnr grid of {n_steps} steps needs r_start > r_min = {r_min}, got {r_start}")
    la, lb = log_snr(min(r_start, 1.0 - r_min)), log_snr(r_min)
    grid = [ratio_of_log_snr(la + (lb - la) * k / (n_steps - 1)) for k in range(n_steps)] + [0.0]
    grid[0] = r_start
    return grid


def log_snr(r):
    """lambda(r) = ln((1 - r)/r)/2: -inf at r = 1, +inf at r = 0."""
    r = float(r)
    if r >= 1.0:
        return -math.inf
    if r <= 0.0:
        return math.inf
    return 0.5 * math.log((1.0 - r) / r)


def ratio_of_log_snr(lam):
    """The inverse of log_snr: r = 1/(1 + e^{2 lambda})."""
    return 1.0 / (1.0 + math.exp(2.0 * lam))


def posterior_coeffs(r_i, r_prev, eta):
    """Coefficients (k_xi, k_x0, sigma) of x_prev = k_xi*x_i + k_x0*x0_hat + sigma*z for
    x_prev = sqrt(1-r_prev) x0_hat + sqrt(r_prev - sigma^2) eps_hat + sigma z,
    eps_hat = (x_i - sqrt(1-r_i) x0_hat)/sqrt(r_i), sigma = eta*sqrt(r_prev/r_i)*sqrt(1-(1-r_i)/(1-r_prev))."""
    if r_prev <= 0.0:
        return 0.0, 1.0, 0.0
    var_ratio = 1.0 if r_i >= 1.0 else 1.0 - (1.0 - r_i) / (1.0 - r_prev)
    sigma = eta * math.sqrt(r_prev / r_i) * math.sqrt(max(var_ratio, 0.0))
    c_eps = math.sqrt(max(r_prev - sigma * sigma, 0.0))
    k_xi = c_eps / math.sqrt(r_i)
    k_x0 = math.sqrt(1.0 - r_prev) - c_eps * math.sqrt(1.0 - r_i) / math.sqrt(r_i)
    return k_xi, k_x0, sigma


def posterior_coef_table(grid, eta):
    """Rows (k_xi, k_x0, sigma, r_prev) of the sampler's device coefficient table, one per step i from grid[i] to
    grid[i + 1].  A step from ratio 0 returns x0_hat (the single-pass case); r_prev is the ratio the masked update noises
    the source to (0 at the last step: the known region is the source itself)."""
    rows = []
    for i in range(len(grid) - 1):
        if grid[i] <= 0.0:
            rows.append((0.0, 1.0, 0.0, 0.0))
        else:
            rows.append(posterior_coeffs(grid[i], grid[i + 1], eta) + (max(float(grid[i + 1]), 0.0),))
    return rows


def dpmpp_2m_coeffs(r_before, r_i, r_prev, eta):
    """(k_xi, k_x0, sigma, c) of the second-order multistep (DPM-Solver++ 2M) step from r_i to r_prev = r_t, whose
    previous step started at r_before (None on the first step):
        D = x0_hat + c*(x0_hat - x0_hat of the previous step),   x_t = k_xi*x_i + k_x0*D + sigma*z
        k_xi = (s_t/s_i) e^{-eta h},  k_x0 = alpha_t (1 - e^{-(1+eta) h}),  sigma = s_t sqrt(1 - e^{-2 eta h}),
        c = h/(2 h_before),  h = lambda(r_t) - lambda(r_i),  h_before = lambda(r_i) - lambda(r_before)
    with alpha = sqrt(1 - r), s = sqrt(r), lambda = log_snr.  This is k-diffusion's dpmpp_2m at eta = 0 and its
    dpmpp_2m_sde (midpoint) at eta > 0.  At eta = 0 and eta = 1, (k_xi, k_x0, sigma) equal posterior_coeffs (DDIM and
    DDPM ancestral); for 0 < eta < 1 it is k-diffusion's family of noise levels, not the DDIM-eta one.  c = 0 (the
    first-order update) on the first step and where h or h_before is infinite (from r = 1, the step after it, the step to
    r = 0).  A step to r_t = 0, or from r_i = 0, returns x0_hat: (0, 1, 0, 0)."""
    r_i, r_t, eta = float(r_i), float(r_prev), float(eta)
    if r_t <= 0.0 or r_i <= 0.0:
        return 0.0, 1.0, 0.0, 0.0
    h = log_snr(r_t) - log_snr(r_i)
    a_t, s_t = math.sqrt(1.0 - r_t), math.sqrt(r_t)
    if math.isinf(h):                          # from r_i = 1: s_i = 1 and every e^{-k h} with k > 0 is 0
        k_xi = s_t if eta == 0.0 else 0.0
        k_x0 = a_t
        sigma = s_t if eta > 0.0 else 0.0
    else:
        k_xi = s_t / math.sqrt(r_i) * math.exp(-eta * h)
        k_x0 = -a_t * math.expm1(-(1.0 + eta) * h)
        sigma = s_t * math.sqrt(-math.expm1(-2.0 * eta * h))
    c = 0.0
    if r_before is not None:
        h_before = log_snr(r_i) - log_snr(r_before)
        if math.isfinite(h) and math.isfinite(h_before) and h_before != 0.0:
            c = h / (2.0 * h_before)
    return k_xi, k_x0, sigma, c


def dpmpp_2m_coef_table(grid, eta):
    """Rows (k_xi, k_x0, sigma, r_prev, c) of the 2M sampler's device coefficient table, one per step i from grid[i] to
    grid[i + 1]: posterior_coef_table's four columns with dpmpp_2m_coeffs's coefficients, and c.  The last row is
    (0, 1, 0, 0, 0) (x0_hat), as is every row of a grid of zeros."""
    rows = []
    for i in range(len(grid) - 1):
        if grid[i] <= 0.0:
            rows.append((0.0, 1.0, 0.0, 0.0, 0.0))
            continue
        k_xi, k_x0, sigma, c = dpmpp_2m_coeffs(grid[i - 1] if i > 0 else None, grid[i], grid[i + 1], eta)
        rows.append((k_xi, k_x0, sigma, max(float(grid[i + 1]), 0.0), c))
    return rows


def normalize_mask(mask, batch, height, width):
    """An inpainting mask as the contiguous float32 [B,1,H,W] buffer the masked posterior reads (1 = generate, 0 = keep,
    fractions feather; the kernel clamps to [0, 1]).  Accepts [H,W], [1,1,H,W] or [B,1,H,W], float32 or bool, on any
    device (the result stays there)."""
    if not torch.is_tensor(mask):
        raise TypeError(f"mask must be a torch tensor, got {type(mask).__name__}")
    if mask.dtype not in (torch.float32, torch.bool):
        raise TypeError(f"mask must be float32 or bool, got {mask.dtype}")
    shape = tuple(mask.shape)
    if shape not in ((height, width), (1, 1, height, width), (batch, 1, height, width)):
        raise ValueError(f"mask of shape {shape} does not broadcast to [{batch},1,{height},{width}]: "
                         f"give [H,W], [1,1,H,W] or [B,1,H,W]")
    return mask.reshape(-1, 1, height, width).expand(batch, 1, height, width).to(torch.float32).contiguous()


def posterior_step_(x_i, x0_hat, r_i, r_prev, z=None, eta=0.0, seed=0, offset=0, src=None, mask=None, known_noise=None):
    """In-place posterior update of x_i (one fused kernel).
    With `mask` (see normalize_mask) and `src` ([B,3,H,W] like x_i): x_i = m*post + (1 - m)*known, known = src noised to
    r_prev = sqrt(1 - r_prev)*src + sqrt(r_prev)*known_noise — replacement inpainting; where m == 0 the result is
    q_sample(src, fixed_r=r_prev, noise=known_noise) bit for bit, src itself at r_prev = 0.  known_noise=None draws it
    in-kernel from its own Philox stream of (seed, offset).  x0_hat may be x_i itself."""
    _require_cuda_f32(x_i, "x_i")
    if not x_i.is_contiguous() or not x0_hat.is_contiguous():
        raise ValueError("posterior_step_ needs contiguous tensors")
    k_xi, k_x0, sigma = posterior_coeffs(float(r_i), float(r_prev), eta)
    masked, _keep = _masked_fields(x_i, r_prev, src, mask, known_noise)
    op = make_op(_lib.OP_POSTERIOR, n=x_i.numel(), x=x_i.data_ptr(), x0_hat=x0_hat.data_ptr(),
                 z=None if z is None else z.contiguous().data_ptr(), k_xi=k_xi, k_x0=k_x0, sigma=sigma,
                 seed=int(seed), offset=int(offset), **masked)
    _lib.run_single(op, _stream(x_i))
    return x_i


def dpmpp_2m_step_(x_i, x0_hat, x0_prev, r_before, r_i, r_prev, z=None, eta=0.0, seed=0, offset=0, src=None, mask=None,
                   known_noise=None):
    """In-place second-order multistep (DPM-Solver++ 2M) update of x_i from r_i to r_prev, one fused kernel: x0_hat is
    extrapolated with the previous step's, x0_prev (r_before: that step's start ratio, None on the first step), with the
    coefficients of dpmpp_2m_coeffs; then x0_prev <- x0_hat for the next step.  Where c = 0 x0_prev is not read (any
    contents), and the result is posterior_step_'s with the same coefficients.  z, seed, offset and the masked form
    (src, mask, known_noise; all-0 mask vectors leave x0_prev as it is) are posterior_step_'s.  x0_hat may be x_i
    itself; x0_prev must be a buffer of its own."""
    _require_cuda_f32(x_i, "x_i")
    if not x_i.is_contiguous() or not x0_hat.is_contiguous():
        raise ValueError("dpmpp_2m_step_ needs contiguous tensors")
    if (not torch.is_tensor(x0_prev) or x0_prev.dtype != torch.float32 or x0_prev.shape != x_i.shape
            or x0_prev.device != x_i.device or not x0_prev.is_contiguous()):
        raise ValueError(f"x0_prev must be a contiguous float32 tensor of x_i's shape {tuple(x_i.shape)} on {x_i.device}")
    if x0_prev.data_ptr() in (x0_hat.data_ptr(), x_i.data_ptr()):
        raise ValueError("x0_prev must not alias x0_hat or x_i")
    k_xi, k_x0, sigma, c = dpmpp_2m_coeffs(r_before, float(r_i), float(r_prev), eta)
    masked, _keep = _masked_fields(x_i, r_prev, src, mask, known_noise)
    op = make_op(_lib.OP_POSTERIOR_2M, x0_prev=x0_prev.data_ptr(), c=c,
                 base=dict(n=x_i.numel(), x=x_i.data_ptr(), x0_hat=x0_hat.data_ptr(),
                           z=None if z is None else z.contiguous().data_ptr(), k_xi=k_xi, k_x0=k_x0, sigma=sigma,
                           seed=int(seed), offset=int(offset), **masked))
    _lib.run_single(op, _stream(x_i))
    return x_i


def _masked_fields(x_i, r_prev, src, mask, known_noise):
    """The masked-form fields of d3fk_posterior_params for posterior_step_ / dpmpp_2m_step_ (empty without a mask), and
    the tensors they point at, which the caller keeps alive until the launch is enqueued."""
    masked = {}
    if mask is None:
        if src is not None or known_noise is not None:
            raise ValueError("posterior_step_: src and known_noise are the masked update's inputs; give a mask with them")
    else:
        if x_i.dim() != 4:
            raise ValueError(f"the masked posterior needs x_i of shape [B,C,H,W], got {tuple(x_i.shape)}")
        B, _, H, W = x_i.shape
        r_prev_k = max(float(r_prev), 0.0)
        if r_prev_k > 1.0:
            raise ValueError(f"r_prev must lie in [0, 1], got {r_prev}")
        if src is None:
            raise ValueError("posterior_step_: a mask needs the source image `src`")
        for name, t in (("src", src), ("known_noise", known_noise)):
            if t is None:
                continue
            if t.dtype != torch.float32:
                raise TypeError(f"{name} must be float32, got {t.dtype}")
            if t.shape != x_i.shape or t.device != x_i.device:
                raise ValueError(f"{name} must have x_i's shape {tuple(x_i.shape)} and device {x_i.device}, "
                                 f"got {tuple(t.shape)} on {t.device}")
        if mask.device != x_i.device:
            raise ValueError(f"mask must be on {x_i.device}, got {mask.device}")
        src = src.contiguous()
        mask = normalize_mask(mask, B, H, W)
        known_noise = None if known_noise is None else known_noise.contiguous()
        masked = dict(r_prev=r_prev_k, src=src.data_ptr(), mask=mask.data_ptr(),
                      known_noise=None if known_noise is None else known_noise.data_ptr(), chw=x_i[0].numel(), hw=H * W)
    return masked, (src, mask, known_noise)


def adam_scalars(lr, beta1, beta2, step, ema_decay=0.0):
    """The per-step scalars of d3fk_adam: (lr, bias1, bias2, ema_decay)."""
    return float(lr), 1.0 - beta1 ** step, 1.0 - beta2 ** step, float(ema_decay)


def adam_step_(p, g, m, v, lr, beta1, beta2, eps, step, ema=None, ema_decay=0.0, grad_scale=1.0, dyn=None):
    """Fused torch.optim.Adam update (+optional EMA lerp) over flat fp32 arenas.  dyn: device float tensor holding
    adam_scalars(...) — the launch then reads its per-step scalars from there (CUDA-graph replay)."""
    _require_cuda_f32(p, "p")
    op = make_op(_lib.OP_ADAM, n=p.numel(), p=p.data_ptr(), g=g.data_ptr(), m=m.data_ptr(), v=v.data_ptr(),
                 ema=None if ema is None else ema.data_ptr(), lr=float(lr), beta1=float(beta1), beta2=float(beta2),
                 eps=float(eps), bias1=1.0 - beta1 ** step, bias2=1.0 - beta2 ** step, ema_decay=float(ema_decay),
                 grad_scale=float(grad_scale), dyn=None if dyn is None else dyn.data_ptr())
    _lib.run_single(op, _stream(p))


def _frames_op(kind, frames, tensor, mean, std):
    N, H, W, _ = frames.shape
    op = make_op(kind, N=N, H=H, W=W, frames=frames.data_ptr(), tensor=tensor.data_ptr(),
                 mean=[float(v) for v in mean], std=[float(v) for v in std])
    _lib.run_single(op, _stream(tensor))


def frames_to_tensor(frames_bgr, mean, std):
    """LitModule.cv2_to_tensor_normalised (d3f/train_deep_fake/lit_module.py:272-283), batched and on the device:
    uint8 BGR frames [N,H,W,3] (or one [H,W,3]) -> normalised fp32 RGB [N,3,H,W] = (v - mean*255) / (std*255)."""
    if frames_bgr.dim() == 3:
        frames_bgr = frames_bgr.unsqueeze(0)
    if not frames_bgr.is_cuda:
        raise _lib.D3fkError("frames must be on a B200 (sm_100a) CUDA device; there is no CPU path")
    if frames_bgr.dtype != torch.uint8 or frames_bgr.dim() != 4 or frames_bgr.shape[-1] != 3:
        raise RuntimeError(f"expected uint8 BGR frames [N,H,W,3], got {frames_bgr.dtype} {tuple(frames_bgr.shape)}")
    frames_bgr = frames_bgr.contiguous()
    N, H, W, _ = frames_bgr.shape
    _lib.init(frames_bgr.device.index if frames_bgr.device.index is not None else torch.cuda.current_device())
    out = torch.empty((N, 3, H, W), dtype=torch.float32, device=frames_bgr.device)
    _frames_op(_lib.OP_FRAMES_TO_TENSOR, frames_bgr, out, mean, std)
    return out


def tensor_to_frames(tensor, mean, std):
    """LitModule.tensor_cv2_to_denormalised (d3f/train_deep_fake/lit_module.py:285-300), batched and on the device:
    fp32 RGB [N,3,H,W] -> uint8 BGR frames [N,H,W,3] = clamp(int(t*std*255 + mean*255), 0, 255).  The input is left
    untouched (the reference scales it in place)."""
    _require_cuda_f32(tensor, "tensor")
    if tensor.dim() != 4 or tensor.shape[1] != 3:
        raise RuntimeError(f"expected fp32 RGB [N,3,H,W], got {tuple(tensor.shape)}")
    tensor = tensor.contiguous()
    N, _, H, W = tensor.shape
    out = torch.empty((N, H, W, 3), dtype=torch.uint8, device=tensor.device)
    _frames_op(_lib.OP_TENSOR_TO_FRAMES, out, tensor, mean, std)
    return out


def random_affine_inverse_maps(B, H, W, degrees=15.0, translate=(0.2, 0.2), scale=(0.8, 1.2), generator=None, device=None,
                               p=1.0):
    """Per-sample inverse affine maps [B,6] (output pixel -> source pixel) with the parameter distribution of the reference's
    `K.RandomAffine(degrees=15, translate=[0.2, 0.2], scale=[0.8, 1.2], shear=0, p=1.0)`
    (d3f/train_denoiser/lit_module.py:55-65): angle ~ U(-degrees, degrees), translation ~ U(-t*W, t*W) x U(-t*H, t*H), one
    isotropic scale ~ U(lo, hi); rotation + scale about the image centre ((W-1)/2, (H-1)/2), then the translation.  Host
    arithmetic on B x 4 numbers (float64, closed-form inverse); the warp itself is d3fk_affine_q_sample.
    p < 1: each sample is augmented with probability p and gets the identity map otherwise (albumentations'
    ShiftScaleRotate(p=0.7) of d3f/train_deep_fake/lit_module.py:99-111; one extra uniform draw per sample)."""
    u = torch.rand(B, 4, generator=generator, dtype=torch.float64)
    keep = torch.rand(B, generator=generator, dtype=torch.float64) < p if p < 1.0 else None
    th = (2 * u[:, 0] - 1) * degrees * math.pi / 180.0
    tx = (2 * u[:, 1] - 1) * translate[0] * W
    ty = (2 * u[:, 2] - 1) * translate[1] * H
    sc = scale[0] + u[:, 3] * (scale[1] - scale[0])
    cx, cy = (W - 1) / 2.0, (H - 1) / 2.0
    # forward: p_out = s R (p_src - c) + c + t, R = [[cos, sin], [-sin, cos]]  =>  p_src = R^T (p_out - c - t) / s + c
    ca, sa = torch.cos(th) / sc, torch.sin(th) / sc
    m = torch.stack([ca, -sa, cx - ca * (cx + tx) + sa * (cy + ty),
                     sa, ca, cy - sa * (cx + tx) - ca * (cy + ty)], dim=1)
    if keep is not None:
        ident = torch.tensor([1.0, 0.0, 0.0, 0.0, 1.0, 0.0], dtype=torch.float64).expand(B, 6)
        m = torch.where(keep.view(B, 1), m, ident)
    return m.to(torch.float32).to(device) if device is not None else m.to(torch.float32)


def affine_q_sample(batch, inverse_maps, lam, noise=None, y=None, seed=0, offset=0, fixed_r=None, return_aux=False,
                    out=None):
    """The reference's `image = augment(image); image_noisy = blend_noise(image)` (d3f/train_denoiser/lit_module.py:113-115) in
    ONE kernel: per-sample affine warp (bilinear, zero padding; `inverse_maps` [B,6] or [B,2,3], output pixel -> source pixel)
    and the noising of the warped image.  Returns (image_augmented, image_noisy) — the loss target and the network input —
    and with return_aux also the per-sample noise ratio.  Noise is that of `q_sample(image_augmented, ...)` with the same
    seed / offset, bit for bit."""
    _require_cuda_f32(batch, "batch")
    if batch.dim() != 4 or batch.shape[-1] % 4:
        raise RuntimeError(f"expected [B,C,H,W] with W a multiple of 4, got {tuple(batch.shape)}")
    batch = batch.contiguous()
    B, C, H, W = batch.shape
    m = inverse_maps.reshape(B, 6).to(device=batch.device, dtype=torch.float32).contiguous()
    aug, noisy = out if out is not None else (torch.empty_like(batch), torch.empty_like(batch))
    for t in (aug, noisy):
        if t.shape != batch.shape or t.dtype != torch.float32 or not t.is_contiguous() or t.device != batch.device:
            raise ValueError("affine_q_sample: `out` must be two contiguous float32 tensors of the batch's shape on its device")
    r_out = torch.empty(B, dtype=torch.float32, device=batch.device) if return_aux else None
    if noise is not None:
        noise = noise.contiguous()
    if y is not None:
        y = y.reshape(B).contiguous()
    op = make_op(_lib.OP_AFFINE_QSAMPLE, B=B, C=C, H=H, W=W, lam=float(lam), fixed_r=-1.0 if fixed_r is None else float(fixed_r),
                 x=batch.data_ptr(), minv=m.data_ptr(), noise=None if noise is None else noise.data_ptr(),
                 y=None if y is None else y.data_ptr(), out_aug=aug.data_ptr(), out_noisy=noisy.data_ptr(),
                 r_out=None if r_out is None else r_out.data_ptr(), seed=int(seed), offset=int(offset))
    _lib.run_single(op, _stream(batch))
    if return_aux:
        return aug, noisy, r_out.view(B, 1, 1, 1)
    return aug, noisy
