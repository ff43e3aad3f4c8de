"""The fused MSE + (1 - SSIM) criterion (csrc/loss.cu) against a float64 reference with a per-pixel error bound.

Reference.  The value and dL/dprediction come from oracle.MseStructuralSimilarityLoss run in float64 under autograd (the
oracle builds its Gaussian window in the input dtype).  Beside it, `explicit_pass` recomputes the same quantities the way
the kernel forms them: the per-window moments mu_x, mu_y, E[x^2], E[y^2], E[xy] of the clipped, normalised inputs (valid
depthwise conv2d with oracle's gaussian_kernel_1d), the SSIM map ss = S1 * S2 with S1 = A1 / B1, S2 = A2 / B2, its partials
a = d ss / d mu_x, b = d ss / d E[x^2], c = d ss / d E[xy] (loss.cu, step 3), and the transposed pass
dss(p) = sum_{windows w containing p} G(p - w) * (a_w + 2 x_p b_w + y_p c_w) (steps 4-5).  test_explicit_pass_reproduces_autograd
shows that these are the quantities behind the autograd gradient, to 1e-12.

Bound.  A first-order model of the kernel's float32 rounding, built from the float64 quantities, per pixel p:

  |err(p)| <= U * (T_MSE * k_mse * (|pred_p| + |target_p|) + T_SSIM * k_ssim * inside_p * S(p))
  S(p) = sum_w G(p - w) * (|a|_w + 2 x_p |b|_w + y_p |c|_w) * (1 + kappa_w)

|a|, |b|, |c| are envelopes: each partial evaluated with every term taken by magnitude, so a partial that vanishes by
cancellation (prediction equal to target, where a = 0 and 2x b + y c = 0 exactly) keeps the size of the rounding its terms
carry.  kappa_w is the window's sensitivity to a relative rounding of its moments: B2 = (E[x^2] - mu_x^2) + (E[y^2] - mu_y^2)
+ C2 cancels when the window is flat, so a relative moment error eps moves B2 by eps * (E[x^2] + E[y^2] + 2 mu_x^2 + 2 mu_y^2),
i.e. kappa_B2 = (that sum) / B2; likewise kappa_B1 = 2 (mu_x^2 + mu_y^2) / B1.  The loss value gets the matching bound, the MSE
part plus sum_w |ss|_w (1 + kappa_w) / nmap, halved.  Every constant is derived in the table below; none is fitted to an
observed error.  The CPU tests show the bound holds for the float32 oracle (not too tight) and flags three float64 mutations
of the kernel's algorithm at the pixels they move (not too loose).

Clip boundary.  torch's clip(0, 1) passes the gradient on the closed range, so a prediction exactly at lo or hi keeps its
SSIM term.  The clamped-prediction cases put 4 % of the pixels there.  Where float32 and float64 normalisation would disagree
about which side of the boundary a value lies on (1 + 2^-23 normalises to exactly 1 in float32 for the range (-1, 1)), the
case generator moves the value to the middle of the range, so membership is the same in the kernel and the reference.

GPU cases run through `value_and_grad`, the training path.  A failure names the first pixel over its bound as (n, c, h, w),
its 32x32 tile and its position inside the tile, and err / bound."""
import pytest
import torch
import torch.nn.functional as F

import oracle
import denoising_diffusion_deep_fake_b200 as d3
from oracle.loss import gaussian_kernel_1d

DEV = "cuda:0"
TILE = 32                # loss.cu: one block per 32x32 tile of one (n, c) plane
WIN = 11                 # 11-tap window, valid SSIM map of (H - 10) x (W - 10)
C1, C2 = 0.01 ** 2, 0.03 ** 2

# ---- constants (each derived from the kernel's arithmetic in csrc/loss.cu, none fitted to observed errors) ----
U = 2.0 ** -24           # fp32 unit roundoff: one rounding of v errs by at most U * |v|
# Relative error of one filtered moment.  Input normalisation (x - lo) * inv_range: 2 roundings plus 1 for the inexact
# inv_range = 3 per x; x * x doubles that and rounds once: 7; the fp32-rounded window taps: 1; 11 horizontal + 11 vertical
# fmaf of non-negative terms: 22.  7 + 1 + 22 = 30.
T_MOM = 30
# The partials are rational in the moments with B2 up to squared (b = -A1 A2 / (B1 B2^2)) and B1, A1, A2 once: a relative
# moment error eps moves a, b, c by at most (1 + kappa) * eps * 3 times their envelope (first order).
K_AMP = 3
# Roundings in forming a, b, c from the moments (squares, three differences, A1, A2, B1, B2, two reciprocals, S1, S2, and
# the longest partial, a: 2 products, 2 differences, 4 products, 1 sum), bounded by 12 on each relative to its envelope.
T_ABC = 12
# Transposed passes (11 + 11 fmaf), the combination A + 2x Bm + y Cm (2 fmaf and 2x exact -> 3 with slack), k_ssim (nmap
# to float, * inv_range, division: 3), the products k_ssim * inside * dss (2) and the final difference with the MSE term (1).
T_TR = 22 + 3 + 3 + 2 + 1
T_SSIM = K_AMP * T_MOM + T_ABC + T_TR        # 133: every rounding on the SSIM gradient path of one pixel
# MSE gradient term k_mse * (pred - target): the difference (1), k_mse = 1 / ntot (1), the product (1), the final sum (1).
T_MSE = 4
# Loss value.  ss_w = S1 * S2: K_AMP * T_MOM from the moments plus A1, A2, B1, B2, the reciprocals and products (6); sums are
# accumulated in double (their rounding is ~2^-53 per term, negligible).  MSE: d rounded once, squared: 2, slack 1.
T_V_SSIM = K_AMP * T_MOM + 6
T_V_MSE = 3
T_V_OUT = 2              # the final double -> float conversion of the loss (1) with slack (1)

RANGES = [(-1.0, 1.0), (0.0, 1.0), (-0.5, 2.5)]
IMPULSES = lambda H, W: [(0, 0), (31, 31), (32, 32), (H - 11, W - 11), (H - 10, W - 10), (H - 1, W - 1)]   # noqa: E731
CONTENTS = ["smooth", "clamped", "saturated", "flat", "near_equal", "impulses"]
BOUNDARY_CONTENTS = {"clamped"}       # contents with values exactly at lo / hi


# ---------------------------------------------------------------------------------------------------------------------
# case generation (float32 CPU tensors)

def _to_range(v, lo, hi):
    """(-1, 1) units -> [lo, hi] units, in float64, then rounded once to float32."""
    return (lo + (v.double() + 1.0) * ((hi - lo) / 2.0)).float()


def _condition(pred, lo, hi):
    """Move values whose clip membership differs between float32 normalisation (the kernel's (x - lo) * inv_range, the
    float32 oracle's (x - lo) / (hi - lo)) and float64 normalisation to the middle of the range."""
    lo32, hi32 = torch.tensor(lo, dtype=torch.float32), torch.tensor(hi, dtype=torch.float32)
    inv = 1.0 / (hi32 - lo32)
    forms = [(pred - lo32) * inv, (pred - lo32) / (hi32 - lo32), (pred.double() - lo) / (hi - lo)]
    ins = [(f >= 0) & (f <= 1) for f in forms]
    disputed = (ins[0] != ins[2]) | (ins[1] != ins[2])
    return torch.where(disputed, torch.tensor((lo + hi) / 2, dtype=torch.float32), pred)


def make_case(content, shape, lo=-1.0, hi=1.0, seed=0):
    """(prediction, target) float32 CPU tensors of one content kind in value range [lo, hi]."""
    g = torch.Generator().manual_seed(seed)
    B, C, H, W = shape
    smooth = F.avg_pool2d(torch.randn(shape, generator=g), 5, 1, 2).clamp(-1, 1) * 1.5   # the existing test's generator
    noise = torch.randn(shape, generator=g)
    if content == "smooth":
        t, p = smooth, smooth + 0.4 * noise
    elif content == "clamped":
        t, p = smooth, smooth + 0.4 * noise                 # clamped below, in range units: values exactly at lo / hi
    elif content == "saturated":
        t, p = smooth, 4.0 * (smooth + 0.4 * noise)         # most of the prediction far outside the range
    elif content == "flat":                                  # sigma = 0: per-plane constants, C2 dominates B2
        level = torch.rand(B, C, 1, 1, generator=g) * 1.6 - 0.8
        t = level.expand(shape).contiguous()
        p = t + 1e-3 * noise
    elif content == "near_equal":                            # the gradient comes from cancellation
        t, p = smooth * 0.6, smooth * 0.6 + 1e-4 * noise
    elif content == "impulses":                              # one impulse per plane, positions cycled over the planes
        t = smooth * 0.5
        p = t.clone()
        pos = IMPULSES(H, W)
        for k in range(B * C):
            h, w = pos[k % len(pos)]
            n, c = divmod(k, C)
            p[n, c, h, w] += -0.5 if t[n, c, h, w] > 0 else 0.5
    else:
        raise ValueError(content)
    t, p = _to_range(t, lo, hi), _to_range(p, lo, hi)
    if content == "clamped":
        p = p.clamp(lo, hi)
    if content == "flat":
        t = _to_range(level.expand(shape), lo, hi).contiguous()
    return _condition(p, lo, hi).contiguous(), t.contiguous()


# ---------------------------------------------------------------------------------------------------------------------
# float64 reference

def _planes(t):
    B, C, H, W = t.shape
    return t.reshape(B * C, 1, H, W)


def _filt(t, g):
    """valid separable Gaussian: window origin w, sum_k G(k) t[w + k]"""
    return F.conv2d(F.conv2d(t, g.view(1, 1, -1, 1)), g.view(1, 1, 1, -1))


def _filt_t(m, g):
    """the transposed pass: pixel p, sum_w G(p - w) m[w]"""
    return F.conv_transpose2d(F.conv_transpose2d(m, g.view(1, 1, 1, -1)), g.view(1, 1, -1, 1))


def oracle64(pred, target, lo, hi):
    """(loss, dL/dpred) of oracle.MseStructuralSimilarityLoss in float64 under autograd."""
    p = pred.double().clone().requires_grad_(True)
    loss = oracle.MseStructuralSimilarityLoss(lo, hi)(p, target.double())
    loss.backward()
    return loss.item(), p.grad


def explicit_pass(pred, target, lo, hi, inclusive=True, mutate=None):
    """The kernel's algorithm in float64.  Returns value, gradient, the per-pixel gradient bound and the value bound.
    inclusive=False applies an exclusive clip mask; mutate(maps) may alter the (a, b, c) window maps or, with
    stage="transposed", the transposed-pass results (the not-too-loose checks)."""
    B, C, H, W = pred.shape
    g = gaussian_kernel_1d(WIN, 1.5, torch.float64)
    p64, t64 = _planes(pred.double()), _planes(target.double())
    xn = (p64 - lo) / (hi - lo)
    x, y = xn.clamp(0.0, 1.0), ((t64 - lo) / (hi - lo)).clamp(0.0, 1.0)
    inside = (((xn >= 0) & (xn <= 1)) if inclusive else ((xn > 0) & (xn < 1))).double()
    mx, my, exx, eyy, exy = (_filt(v, g) for v in (x, y, x * x, y * y, x * y))
    mxx, myy, mxy = mx * mx, my * my, mx * my
    A1, B1 = 2 * mxy + C1, mxx + myy + C1
    A2, B2 = 2 * (exy - mxy) + C2, (exx - mxx) + (eyy - myy) + C2
    S1, S2 = A1 / B1, A2 / B2
    ss = S1 * S2
    a = S2 * 2 * (my - S1 * mx) / B1 + S1 * 2 * (S2 * mx - my) / B2
    b = -S1 * S2 / B2
    c = 2 * S1 / B2
    if mutate is not None:
        a, b, c = mutate("windows", (a, b, c))
    TA, TB, TC = (_filt_t(m, g) for m in (a, b, c))
    if mutate is not None:
        TA, TB, TC = mutate("transposed", (TA, TB, TC))
    dss = TA + 2 * x * TB + y * TC
    ntot = pred.numel()
    nmap = B * C * (H - WIN + 1) * (W - WIN + 1)
    k_mse, k_ssim = 1.0 / ntot, 0.5 / ((hi - lo) * nmap)
    d = p64 - t64
    grad = k_mse * d - k_ssim * inside * dss
    loss = 0.5 * ((d * d).mean().item() + 1.0 - ss.mean().item())
    # envelopes and conditioning
    eS1 = (2 * mxy.abs() + C1) / B1
    eS2 = (2 * (exy.abs() + mxy.abs()) + C2) / B2
    ea = eS2 * 2 * (my.abs() + eS1 * mx.abs()) / B1 + eS1 * 2 * (eS2 * mx.abs() + my.abs()) / B2
    eb, ec = eS1 * eS2 / B2, 2 * eS1 / B2
    kappa = (exx + eyy + 2 * mxx + 2 * myy) / B2 + 2 * (mxx + myy) / B1
    w1 = 1.0 + kappa
    S = _filt_t(ea * w1, g) + 2 * x * _filt_t(eb * w1, g) + y * _filt_t(ec * w1, g)
    bound = U * (T_MSE * k_mse * (p64.abs() + t64.abs()) + T_SSIM * k_ssim * inside * S)
    vbound = (0.5 * U * (T_V_MSE * (d * d).mean().item() + T_V_SSIM * (eS1 * eS2 * w1).sum().item() / nmap)
              + T_V_OUT * U * abs(loss))
    shape = (B, C, H, W)
    return {"loss": loss, "grad": grad.reshape(shape), "bound": bound.reshape(shape), "vbound": vbound}


# ---------------------------------------------------------------------------------------------------------------------
# checking

def over_bound(err, bound):
    """None when err <= bound everywhere, else a message naming the first pixel over its bound."""
    bad = err > bound
    if not bool(bad.any()):
        return None
    B, C, H, W = err.shape
    k = int(bad.flatten().nonzero()[0])
    n, rem = divmod(k, C * H * W)
    c, rem = divmod(rem, H * W)
    h, w = divmod(rem, W)
    e, bd = err[n, c, h, w].item(), bound[n, c, h, w].item()
    return (f"{int(bad.sum())} of {err.numel()} pixels over the bound; first at (n, c, h, w) = ({n}, {c}, {h}, {w}), "
            f"tile ({h // TILE}, {w // TILE}) position ({h % TILE}, {w % TILE}): err {e:.3e} bound {bd:.3e} "
            f"(err/bound {e / bd:.3g})")


def max_ratio(err, bound):
    return (err / bound).max().item()


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests: the reference and the bound

CPU_SHAPE = (2, 3, 64, 96)


@pytest.mark.parametrize("lo,hi", RANGES)
@pytest.mark.parametrize("content", ["smooth", "clamped", "impulses"])
def test_explicit_pass_reproduces_autograd(content, lo, hi):
    """The explicit pass's partials, pushed through the transposed filter and scaled as loss.cu does, are the float64
    autograd gradient of the oracle: the bound is built from the right quantities."""
    if content in BOUNDARY_CONTENTS and (lo, hi) == (-0.5, 2.5):
        pytest.skip("no exact-boundary contents in the range with an inexact 1 / (hi - lo)")
    pred, target = make_case(content, CPU_SHAPE, lo, hi, seed=1)
    loss, grad = oracle64(pred, target, lo, hi)
    ref = explicit_pass(pred, target, lo, hi)
    scale = grad.abs().max().item()
    assert (ref["grad"] - grad).abs().max().item() <= 1e-12 * scale
    assert abs(ref["loss"] - loss) <= 1e-12


def _cpu_cases():
    cases = [(c, (-1.0, 1.0)) for c in CONTENTS]
    cases += [(c, (0.0, 1.0)) for c in ("smooth", "clamped", "saturated")]
    cases += [(c, (-0.5, 2.5)) for c in ("smooth", "saturated", "flat", "near_equal")]
    return cases


@pytest.mark.parametrize("content,rng", _cpu_cases())
def test_float32_oracle_inside_bound(content, rng):
    """Not too tight: the float32 oracle (a different float32 evaluation of the same criterion) stays inside the bound at
    every pixel, and its value inside the value bound."""
    lo, hi = rng
    pred, target = make_case(content, CPU_SHAPE, lo, hi, seed=2)
    ref = explicit_pass(pred, target, lo, hi)
    p = pred.clone().requires_grad_(True)
    loss32 = oracle.MseStructuralSimilarityLoss(lo, hi)(p, target)
    loss32.backward()
    msg = over_bound((p.grad.double() - ref["grad"]).abs(), ref["bound"])
    assert msg is None, msg
    assert abs(loss32.item() - ref["loss"]) <= ref["vbound"], (loss32.item(), ref["loss"], ref["vbound"])


def _window_zeroed(plane, wr, wc):
    def mutate(stage, maps):
        if stage != "windows":
            return maps
        out = []
        for m in maps:
            m = m.clone()
            m[plane, 0, wr, wc] = 0.0
            out.append(m)
        return out
    return mutate


def _transposed_shifted(col):
    """The transposed-pass result of every tile's column `col` read one pixel to the left (a tile-edge indexing slip)."""
    def mutate(stage, maps):
        if stage != "transposed":
            return maps
        out = []
        for m in maps:
            m = m.clone()
            W = m.shape[-1]
            cols = torch.arange(col, W, TILE)
            m[..., cols] = m[..., cols - 1]
            out.append(m)
        return out
    return mutate


@pytest.mark.parametrize("mutation", ["exclusive_clip", "window_31_31_zeroed", "transposed_shift_col31"])
def test_bound_flags_mutations(mutation):
    """Not too loose: each float64 mutation of the kernel's algorithm is flagged, only at pixels it moves, and a mutation
    that drops or misplaces a whole term is flagged at most pixels it moves."""
    lo, hi = -1.0, 1.0
    pred, target = make_case("clamped" if mutation == "exclusive_clip" else "smooth", CPU_SHAPE, lo, hi, seed=3)
    ref = explicit_pass(pred, target, lo, hi)
    if mutation == "exclusive_clip":
        mut = explicit_pass(pred, target, lo, hi, inclusive=False)
        expect = ((pred == lo) | (pred == hi))
    elif mutation == "window_31_31_zeroed":
        mut = explicit_pass(pred, target, lo, hi, mutate=_window_zeroed(1, 31, 31))
        expect = torch.zeros(pred.shape, dtype=torch.bool)
        expect[0, 1, 31:31 + WIN, 31:31 + WIN] = True
    else:
        mut = explicit_pass(pred, target, lo, hi, mutate=_transposed_shifted(TILE - 1))
        expect = torch.zeros(pred.shape, dtype=torch.bool)
        expect[..., TILE - 1::TILE] = True
    delta = (mut["grad"] - ref["grad"]).abs()
    flagged = delta > ref["bound"]
    assert bool((delta[~expect] == 0).all()), "the mutation moved pixels outside its expected set"
    assert not bool((flagged & ~expect).any())
    assert bool(flagged.any())
    if mutation != "window_31_31_zeroed":
        # a dropped SSIM term is flagged at nearly every pixel it touches, a one-pixel shift of the transposed sums at most
        # of them (neighbouring sums of smooth content are close).  One window of the 121 that cover a pixel moves it by
        # G(p - w) of its partials, which clears the bound only near the window's centre: no fraction asserted there.
        frac = flagged[expect & (delta > 0)].double().mean().item()
        assert frac > {"exclusive_clip": 0.9, "transposed_shift_col31": 0.5}[mutation], frac


def test_clamped_cases_put_pixels_on_the_boundary():
    pred, _ = make_case("clamped", CPU_SHAPE, -1.0, 1.0, seed=0)
    frac = ((pred == -1.0) | (pred == 1.0)).double().mean().item()
    assert 0.02 < frac < 0.2, frac


# ---------------------------------------------------------------------------------------------------------------------
# GPU tests: the kernel against the float64 reference

SMALL = (2, 3, 64, 96)
EDGE_SHAPES = [(1, 1, 32, 32), (2, 3, 32, 96), (2, 3, 96, 32), (1, 3, 256, 256)]   # (1, 1, 32, 32): every tile edge is an image edge
BENCH_SHAPES = [(256, 3, 64, 64), (14, 3, 128, 128), (64, 3, 128, 128)]            # training step; the swap-step plans


def _gpu_cases():
    cases = [(c, SMALL, (-1.0, 1.0)) for c in CONTENTS]
    cases += [(c, SMALL, (0.0, 1.0)) for c in ("smooth", "clamped", "saturated", "impulses")]
    cases += [(c, SMALL, (-0.5, 2.5)) for c in ("smooth", "saturated", "flat", "near_equal", "impulses")]
    cases += [(c, s, (-1.0, 1.0)) for s in EDGE_SHAPES for c in ("smooth", "clamped")]
    cases += [(c, s, (-1.0, 1.0)) for s in BENCH_SHAPES for c in ("smooth", "clamped", "flat")]
    return [pytest.param(c, s, r, id=f"{c}-{'x'.join(map(str, s))}-{r[0]:g}_{r[1]:g}") for c, s, r in cases]


def _workspace_zero():
    ws = d3.loss._workspace(torch.device(DEV))
    torch.cuda.synchronize()
    return bool((ws == 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("content,shape,rng", _gpu_cases())
def test_fused_criterion_against_float64(content, shape, rng):
    lo, hi = rng
    pred, target = make_case(content, shape, lo, hi, seed=4)
    loss64, grad64 = oracle64(pred, target, lo, hi)
    ref = explicit_pass(pred, target, lo, hi)
    crit = d3.MseStructuralSimilarityLoss(lo, hi)
    loss, grad = crit.value_and_grad(pred.to(DEV), target.to(DEV))
    assert _workspace_zero(), "the loss workspace (two sums and the block ticket) was not reset"
    err = (grad.cpu().double() - grad64).abs()
    verr = abs(loss.item() - loss64)
    print(f"criterion {content} {shape} {rng}: max err/bound gradient {max_ratio(err, ref['bound']):.3g} "
          f"value {verr / ref['vbound']:.3g}")
    msg = over_bound(err, ref["bound"])
    assert msg is None, msg
    assert verr <= ref["vbound"], f"loss {loss.item()!r} float64 {loss64!r}: err {verr:.3e} bound {ref['vbound']:.3e}"


def _ulp32(v):
    v = torch.tensor(abs(v), dtype=torch.float32)
    return (torch.nextafter(v, torch.tensor(float("inf"))) - v).item()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(8, 3, 64, 64), (256, 3, 64, 64)])
def test_criterion_paths_agree(shape):
    """The training path (autograd forward + backward(3.0)), value_and_grad, and the forward without a gradient
    (grad == NULL) give the same value within 1 fp32 ulp (the double atomics sum in a varying order); the gradient path
    has no atomics, so consecutive launches give bit-identical gradients and the autograd gradient is exactly 3 times the
    value_and_grad one.  The workspace reads back as zeros after every launch."""
    pred, target = make_case("clamped", shape, seed=5)
    pred, target = pred.to(DEV), target.to(DEV)
    crit = d3.MseStructuralSimilarityLoss(-1.0, 1.0)
    pd = pred.clone().requires_grad_(True)
    l_train = crit(pd, target)
    assert _workspace_zero()
    (l_train * 1.0).backward(torch.tensor(3.0, device=DEV))
    l_nograd = crit(pred, target)
    assert _workspace_zero()
    l1, g1 = crit.value_and_grad(pred, target)
    assert _workspace_zero()
    l2, g2 = crit.value_and_grad(pred, target)
    assert _workspace_zero()
    ulp = _ulp32(l1.item())
    for v in (l_train.item(), l_nograd.item(), l2.item()):
        assert abs(v - l1.item()) <= ulp, (v, l1.item())
    assert torch.equal(g1, g2)
    assert torch.equal(pd.grad, g1 * 3.0)
