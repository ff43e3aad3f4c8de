"""GPU suite (-m gpu): eval-mode autograd (the frozen-BN plan) and the input gradient.

Kernel cases are bit-exact on integer-valued data in the style of test_gpu_exact.py: the stem's input-gradient kernel
(stem_dgrad.cu) sums at most 49 * 64 products of integers bounded by 2 x 2, far below 2^21, so its fp32 output equals the
float64 transposed convolution exactly; the frozen BatchNorm backward writes dx = fl(fl(gamma * invstd) * dy') (one fp32
product with the coefficient the kernel forms the same way, then the dtype store), so dx and dres are exact too, and only the
two reduction sums carry a bound (test_gpu_exact.check_bn_bwd_sums).  Whole-network cases compare against the float64
oracle in .eval() and check the module contract (buffers untouched, graph semantics, no growth over an input-gradient loop)."""
import copy

import pytest
import torch
import torch.nn.functional as F

import oracle
import denoising_diffusion_deep_fake_b200 as d3
from denoising_diffusion_deep_fake_b200 import _lib
from test_gpu_exact import (BF16, DTYPES, F32, EXACT_LIMIT, assert_equal, assert_pinned, bn_bwd_inputs, bn_bwd_outputs,   # noqa: F401
                            bn_bwd_fields, check_bn_bwd_sums, check_conv_outputs, declared_classes, launched_classes,
                            op_classes, run, run_conv_case, verbose)
from test_gpu_parity_configs import LAM, cosine, faces, noised, oracle64, product, state_at, trained   # noqa: F401

DEV = "cuda:0"


@pytest.fixture(autouse=True)
def _device():
    if torch.cuda.is_available():
        _lib.init(0)


def rel(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return ((a - b).norm() / (b.norm() + 1e-300)).item()


# ------------------------------------------------------------------ launch classes of the kernels this file adds
def stem_dgrad_class(op):
    """try_launch_stem_dgrad's conditions (the kernel prints no launch line)."""
    p = _lib.op_params(op)
    if (op.kind == _lib.OP_CONV and p.dtype == BF16 and p.mode == 1 and p.kh == 7 and p.kw == 7 and p.stride == 2 and p.pad == 3
            and p.c0 == 64 and p.c1 == 0 and 1 <= p.Cout <= 3 and p.out_nchw and not p.out and not p.res and not p.stats
            and not p.relu and not p.scale and not p.shift and not p.bw_x and p.Ho == 2 * p.Hi and p.Wo == 2 * p.Wi
            and p.Ho % 32 == 0 and p.Wo % 32 == 0 and p.ld0 % 8 == 0):
        return ["stem_dgrad"]
    return []


def frozen_bn_classes(op):
    p = _lib.op_params(op)
    if op.kind not in (_lib.OP_BN_BWD, _lib.OP_BN_BWD_APPLY) or not p.frozen:
        return []
    dt = {F32: "f32", BF16: "bf16"}[p.dtype]
    xm = int(bool(p.relu and p.mask_from_x))
    if op.kind == _lib.OP_BN_BWD:
        return [f"bn_bwd_frozen<{dt}> xmask={xm}", "bn_bwd_finalize"]
    return [f"bn_bwd_apply<{dt}> xmask={xm} frozen"]


PINNED_HERE = {"stem_dgrad", "bn_bwd_finalize"} | {f"bn_bwd_frozen<{d}> xmask={x}" for d in ("f32", "bf16") for x in (0, 1)} | \
    {f"bn_bwd_apply<{d}> xmask={x} frozen" for d in ("f32", "bf16") for x in (0, 1)}


# ------------------------------------------------------------------ stem input gradient, bit-exact
STEM_DGRAD_CASES = [(B, H, W) for B in (1, 3, 256) for H, W in ((64, 64), (128, 128), (32, 96), (96, 96), (256, 256))]


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,W", STEM_DGRAD_CASES)
def test_stem_dgrad_exact(B, H, W):
    """dX = conv_transpose2d(dY, w, stride 2, pad 3, output_padding 1), fp32 NCHW, equal to float64 at every pixel: both output
    parities at every image edge (and the 32 x 32 tile edges in between) are in the comparison."""
    g = torch.Generator().manual_seed(B * 7 + H + W)
    Hy, Wy = H // 2, W // 2
    dy = torch.randint(-2, 3, (B, Hy, Wy, 64), generator=g).float()
    w = torch.randint(-2, 3, (3, 7, 7, 64), generator=g).float()
    assert 49 * 64 * 2 * 2 < EXACT_LIMIT
    dy_d = dy.to(DEV).to(torch.bfloat16)
    w_d = w.to(DEV).to(torch.bfloat16).contiguous()
    out = torch.full((B, 3, H, W), float("nan"), device=DEV)
    op = _lib.make_op(_lib.OP_CONV, dtype=BF16, mode=1, src0=dy_d.data_ptr(), c0=64, ld0=64, B=B, Hi=Hy, Wi=Wy, Ho=H, Wo=W,
                      kh=7, kw=7, stride=2, pad=3, w=w_d.data_ptr(), Cout=3, out_nchw=out.data_ptr())
    assert stem_dgrad_class(op) == ["stem_dgrad"]
    run(op)
    ref = F.conv_transpose2d(dy.to(DEV).double().permute(0, 3, 1, 2), w.to(DEV).double().permute(3, 0, 1, 2), stride=2, padding=3,
                             output_padding=1)
    assert_equal(out, ref, f"stem dgrad B={B} {H}x{W}", "nchw")


# ------------------------------------------------------------------ frozen BatchNorm backward, bit-exact dx
FROZEN_BN_CASES = [(64, 2 * 32 * 32), (128, 3000), (512, 64), (32, 50000)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C,count", FROZEN_BN_CASES)
@pytest.mark.parametrize("kind", ["single_pass", "apply"])
@pytest.mark.parametrize("mask_from_x,dres", [(1, False), (0, False), (0, True)])
def test_frozen_bn_bwd_exact(dtype, C, count, kind, mask_from_x, dres):
    """D3FK_OP_BN_BWD with `frozen` (the one-pass kernel + bn_bwd_finalize) and D3FK_OP_BN_BWD_APPLY with `frozen` (after a
    dgrad that fused the sums: here the sums are given): dx = A * dy' and dres = dy' exactly, dgamma / dbeta = the sums."""
    d = bn_bwd_inputs(dtype, C, count, 4000 + C + count)
    o = bn_bwd_outputs(dtype, C, count)
    f = bn_bwd_fields(dtype, C, count, d, mask_from_x, o)
    f.update(frozen=1)
    if not dres:
        f.update(dres=None)
    gp = d["dy"].double() * d["mask"]
    xhat = (d["x"].double() - d["mean"].double()) * d["invstd"].double()
    if kind == "apply":
        o["bstats"][0] = gp.sum(0)
        o["bstats"][1] = (gp * xhat).sum(0)
        op = _lib.make_op(_lib.OP_BN_BWD_APPLY, **f)
    else:
        f.update(coef=None)
        op = _lib.make_op(_lib.OP_BN_BWD, **f)
    run(op)
    A = d["gamma"] * d["invstd"]
    assert_equal(o["dx"], (A.double() * gp).float(), f"frozen {kind} dx", "pc")
    if dres:
        assert_equal(o["dres"], gp, f"frozen {kind} dres", "pc")
    else:
        assert float(o["dres"].abs().max()) == 0.0
    if kind == "single_pass":
        check_bn_bwd_sums(o["bstats"], gp, xhat, f"frozen {kind}")
    assert_equal(o["dbeta"], o["bstats"][0].float(), "dbeta", "c")
    assert_equal(o["dgamma"], o["bstats"][1].float(), "dgamma", "c")
    assert _lib.load().d3fk_device_error_flag() == 0


@pytest.mark.gpu
def test_bn_fold_publishes_running_statistics():
    C = 64
    rm, rv = torch.randn(C, device=DEV), torch.rand(C, device=DEV) + 0.5
    gamma, beta = torch.rand(C, device=DEV) + 0.5, torch.randn(C, device=DEV)
    sc, sh, mean, invstd = (torch.zeros(C, device=DEV) for _ in range(4))
    run(_lib.make_op(_lib.OP_BN_FOLD, dtype=F32, C=C, eps=1e-5, gamma=gamma.data_ptr(), beta=beta.data_ptr(),
                     running_mean=rm.data_ptr(), running_var=rv.data_ptr(), scale=sc.data_ptr(), shift=sh.data_ptr(),
                     mean=mean.data_ptr(), invstd=invstd.data_ptr()))
    assert torch.equal(mean, rm)
    assert torch.equal(invstd, 1.0 / torch.sqrt(rv + 1e-5)) or rel(invstd, 1.0 / torch.sqrt(rv.double() + 1e-5)) < 1e-7
    assert torch.equal(sc, gamma * invstd)


# ------------------------------------------------------------------ the frozen plan's forward convolution without epilogue
# (raw output kept for the BN apply pass: no statistics, no scale / shift) on the TMA-fed generic path, one K slice
FROZEN_CONV_CASES = [dict(B=256, Hi=8, Wi=8, c0=128, c1=0, up0=0, Cout=128, k=3, stride=1, pad=1, mode=0,
                          pin={"conv<128,2> mode=0 KS=1 epi=0"})]


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(FROZEN_CONV_CASES)))
def test_frozen_forward_conv_exact(verbose, capfd, i):
    c = FROZEN_CONV_CASES[i]
    g, o, v = run_conv_case(BF16, c, seed=900 + i)
    check_conv_outputs(c, g, o, v, f"FROZEN_CONV_CASES[{i}]")
    assert_pinned(capfd, c["pin"])


# ------------------------------------------------------------------ launch classes of the new plans
@pytest.mark.gpu
def test_new_plans_launch_only_pinned_classes(verbose, capfd):
    """One eval-mode forward + backward (frozen-BN plan, with and without dX) and one training step with dX at the
    benchmarked shapes: every launched class is pinned by test_gpu_exact.py or by a case of this file."""
    torch.manual_seed(0)
    m = d3.Unet(precision="bf16").to(DEV)
    seen = set()
    capfd.readouterr()
    for training, B, H, want_dx in ((False, 64, 128, True), (False, 256, 64, False), (True, 256, 64, True)):
        m.train(training)
        x = torch.randn(B, 3, H, H, device=DEV).clamp(-1, 1).requires_grad_(want_dx)
        y = m(x)
        y.backward(torch.randn_like(y))
        torch.cuda.synchronize()
        seen |= set(launched_classes(capfd.readouterr().err))
    for plans in m._plans.values():
        for plan in plans:
            for ol in [plan.pack_ops, plan.fwd_ops] + list(plan.bwd_segments or []):
                for op in ol:
                    seen |= set(stem_dgrad_class(op)) | set(frozen_bn_classes(op))
                    if not frozen_bn_classes(op):
                        seen |= set(op_classes(op))
    assert "stem_dgrad" in seen and "bn_bwd_frozen<bf16> xmask=1" in seen
    missing = seen - declared_classes() - PINNED_HERE - set().union(*(c["pin"] for c in FROZEN_CONV_CASES))
    assert not missing, f"classes the new plans launch but no exact case pins: {sorted(missing)}"


# ------------------------------------------------------------------ whole network against the float64 oracle
def _grads(trained, precision, B, H, train, seeds):
    """Parameter gradients and x.grad of one loss (noising -> U-Net -> MSE+SSIM) in the given mode: d3fk (`precision`), the
    float64 oracle, and torch's own run of the oracle in that precision on this GPU (fp32 with TF32 off / bf16 autocast) —
    the yardstick test_gpu_parity_configs uses for inputs on which the trained network itself is ill-conditioned."""
    ref, _ = trained
    sd = state_at(trained, H)
    x0 = faces(B, H, H, seeds[0])
    noise, y = noised(x0, seeds[1])
    noisy = d3.q_sample(x0, LAM, noise=noise, y=y)
    m = product(precision, sd, train)
    xin = noisy.clone().requires_grad_()
    d3.MseStructuralSimilarityLoss(-1.0, 1.0)(m(xin), x0).backward()
    crit64 = oracle.MseStructuralSimilarityLoss(-1.0, 1.0)
    r64 = oracle64(ref, sd, train)
    x64 = noisy.double().clone().requires_grad_()
    crit64(r64(x64), x0.double()).backward()
    lib = copy.deepcopy(ref)
    lib.load_state_dict(sd)
    lib = lib.to(DEV).train(train)
    amp = precision == "bf16"
    if amp:
        lib = lib.to(memory_format=torch.channels_last)
    xl = (noisy.contiguous(memory_format=torch.channels_last) if amp else noisy.clone()).requires_grad_()
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
        pred_lib = lib(xl)
    crit64(pred_lib.float(), x0).backward()
    grads = lambda mod, x: ({n: p.grad for n, p in mod.named_parameters()}, x.grad)
    return m, grads(m, xin), grads(r64, x64), grads(lib, xl)


def _distances(m, src, ref64):
    """Norm-relative distance to the float64 oracle: whole arena, each of the five buckets, x.grad."""
    (g, dx), (g64, dx64) = src, ref64
    names = m._param_names
    cat = lambda d, sel: torch.cat([d[n].flatten().double() for n in sel])
    out = {"arena": rel(cat(g, names), cat(g64, names)), "x.grad": rel(dx, dx64)}
    for i, (s0, s1) in enumerate(m.grad_buckets()):
        sel = [n for n in names if s0 <= m._grad_offsets[n] < s1]
        out[f"bucket{i}"] = rel(cat(g, sel), cat(g64, sel))
    return out


def _check_draws(trained, precision, B, H, train, tol_arena, tol_bucket):
    """The bounds of test_gpu_parity_configs.test_train_step_gradients_benchmarked_configs: arena within tol_arena, each bucket
    within tol_bucket — or within 1.5x (fp32) / 2x (bf16) torch's own distance, whichever is larger; x.grad is held to the
    bucket bound.  bf16: up to three input draws, the first that satisfies every bound passes (a wrong layer fails every draw)."""
    draws = [(21, 23), (31, 33), (41, 43)] if precision == "bf16" else [(21, 23)]
    factor = 2.0 if precision == "bf16" else 1.5
    history = []
    for seeds in draws:
        m, mine, ref64, lib = _grads(trained, precision, B, H, train, seeds)
        e, e_lib = _distances(m, mine, ref64), _distances(m, lib, ref64)
        bad = [k for k in e if e[k] > max(tol_arena if k == "arena" else tol_bucket, factor * e_lib[k])]
        history.append(", ".join(f"{k} {e[k]:.2e} (torch {e_lib[k]:.2e})" for k in e))
        print(seeds, history[-1], "cos x.grad", f"{cosine(mine[1], ref64[1]):.8f}")
        if not bad:
            return
    raise AssertionError("no draw within the bounds:\n" + "\n".join(history))


@pytest.mark.gpu
@pytest.mark.parametrize("precision,B,H,tol_arena,tol_bucket", [
    ("fp32", 8, 64, 1e-5, 1e-4), ("fp32", 256, 64, 1e-5, 1e-4),
    ("bf16", 8, 64, 2e-2, 5e-2), ("bf16", 256, 64, 2e-2, 5e-2), ("bf16", 64, 128, 2e-2, 5e-2),
])
def test_eval_gradients_vs_oracle(trained, precision, B, H, tol_arena, tol_bucket):
    """Eval mode (BatchNorm on the running statistics, trained weights): every parameter gradient and x.grad against the
    float64 oracle in .eval()."""
    _check_draws(trained, precision, B, H, False, tol_arena, tol_bucket)


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol_arena,tol_bucket", [("fp32", 1e-5, 1e-4), ("bf16", 2e-2, 5e-2)])
def test_train_input_gradient_vs_oracle(trained, precision, tol_arena, tol_bucket):
    """Training mode with x.requires_grad (the training plan with the stem dgrad): gradients and x.grad against the oracle."""
    _check_draws(trained, precision, 8, 64, True, tol_arena, tol_bucket)


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp32", 2e-5), ("bf16", 3e-2)])
def test_frozen_backward_in_situ(precision, tol):
    """Flip-free: the GPU frozen plan's forward buffers copied into a CPU twin whose backward the interpreter runs (frozen BN
    semantics of test_grad_modes_cpu), both backwards see identical masks; parameter gradients and dX must agree."""
    import op_interpreter as I
    from denoising_diffusion_deep_fake_b200.plan import UnetPlan
    import test_grad_modes_cpu as T
    torch.manual_seed(5)
    ref, m = T.make_pair(seed=5)
    m = m if precision == "fp32" else d3.Unet(precision="bf16")
    m.load_state_dict(ref.state_dict())
    m = m.to(DEV).eval()
    B, H, W = 16, 64, 64
    x = torch.randn(B, 3, H, W)
    dy = torch.randn(B, 3, H, W)
    xin = x.to(DEV).requires_grad_()
    m(xin).backward(dy.to(DEV))
    torch.cuda.synchronize()
    plan = next(p for plans in m._plans.values() for p in plans if p.frozen)
    mc = d3.Unet(precision="fp32")
    mc.load_state_dict({k: v.cpu() for k, v in m.state_dict().items()})
    twin = T.cpu_plan(mc, B, H, W, False, frozen=True, want_dx=True)
    only_gpu = [plan.ws, getattr(plan, "w_stem_s2d", None), getattr(plan, "xs2d", None)]
    gpu_keep = [t for t in plan.keep if not any(t is o for o in only_gpu)]
    assert len(twin.keep) == len(gpu_keep)
    for tc, tg in zip(twin.keep, gpu_keep):
        if tc.shape == tg.shape:
            tc.copy_(tg.to("cpu").to(tc.dtype))
    twin.x8.t.zero_()
    twin.x8.t[..., :3] = x.permute(0, 2, 3, 1)
    saved = dict(I._DISPATCH)
    I._DISPATCH.update({_lib.OP_BN_FOLD: T._run_bn_fold, _lib.OP_BN_BWD: T._run_bn_bwd, _lib.OP_BN_BWD_APPLY: T._run_bn_bwd_apply})
    try:
        dx = torch.empty_like(x)
        T.run_backward(twin, dy, dx)
    finally:
        I._DISPATCH.clear()
        I._DISPATCH.update(saved)
    a = torch.cat([p.grad.cpu().flatten() for n, p in sorted(m.named_parameters())])
    b = torch.cat([mc._grad_arena[mc._grad_offsets[n]:mc._grad_offsets[n] + p.numel()] for n, p in sorted(m.named_parameters())])
    assert rel(a, b) < tol and rel(xin.grad.cpu(), dx) < tol, (rel(a, b), rel(xin.grad.cpu(), dx))


# ------------------------------------------------------------------ module contract
@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-6), ("bf16", 3e-2)])
def test_eval_contract(precision, tol):
    """BN buffers and parameters bitwise unchanged by an eval-mode forward + backward; the autograd eval forward equals the
    no_grad one.  bf16 bound: the frozen plan stores each of the 46 raw conv outputs in bf16 before its BN apply, the fused eval
    plan does not — one extra round-to-nearest (2^-9 relative) per layer; uncorrelated, they add up to sqrt(46) * 2^-9 = 1.3e-2
    norm-relative before the network's own gain; 3e-2 leaves 2.3x for that gain."""
    torch.manual_seed(0)
    m = d3.Unet(precision=precision).to(DEV)
    with torch.no_grad():
        m.train()
        for _ in range(2):
            m(torch.randn(8, 3, 64, 64, device=DEV))
    m.eval()
    x = torch.randn(4, 3, 64, 64, device=DEV)
    with torch.no_grad():
        y0 = m(x)
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    y = m(x)
    assert y.grad_fn is not None
    assert rel(y.detach(), y0) < tol
    y.square().mean().backward()
    torch.cuda.synchronize()
    for k, v in m.state_dict().items():
        assert torch.equal(v, sd0[k]), k
    # input gradient with every parameter frozen, both modes; accumulation; double backward raises
    for p in m.parameters():
        p.requires_grad_(False)
    for training in (False, True):
        m.train(training)
        xg = x.clone().requires_grad_()
        (gx,) = torch.autograd.grad(m(xg).square().mean(), xg)
        assert gx.shape == x.shape and torch.isfinite(gx).all() and gx.abs().sum() > 0
        m(xg).square().mean().backward()
        g1 = xg.grad.clone()
        m(xg).square().mean().backward()
        if not training:          # eval mode is deterministic: two equal backwards accumulate to exactly twice
            assert torch.equal(xg.grad, 2 * g1)
        (gx,) = torch.autograd.grad(m(xg).square().mean(), xg, create_graph=True)
        with pytest.raises(RuntimeError):
            gx.sum().backward()
    assert _lib.load().d3fk_device_error_flag() == 0


@pytest.mark.gpu
def test_input_gradient_loop_does_not_grow():
    torch.manual_seed(0)
    m = d3.Unet(precision="bf16").to(DEV).eval()
    for p in m.parameters():
        p.requires_grad_(False)
    x = torch.randn(64, 3, 128, 128, device=DEV)

    def step(x):
        xg = x.detach().requires_grad_()
        (g,) = torch.autograd.grad(m(xg).square().mean(), xg)
        return (x - 0.01 * g.sign()).clamp(-1, 1)

    for _ in range(2):
        x = step(x)
    torch.cuda.synchronize()
    n_plans = sum(len(v) for v in m._plans.values())
    mem = torch.cuda.memory_allocated()
    for _ in range(20):
        x = step(x)
    torch.cuda.synchronize()
    assert sum(len(v) for v in m._plans.values()) == n_plans
    assert torch.cuda.memory_allocated() <= mem
    assert _lib.load().d3fk_device_error_flag() == 0
