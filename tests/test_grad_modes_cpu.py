"""CPU suite: eval-mode autograd (the frozen-BN plan) and the input gradient, on the host.

The exact op lists are executed by the torch-CPU interpreter (tests/op_interpreter.py), with its BatchNorm entries extended
here for the `frozen` flag of d3fk_bn_params (backward on the running statistics) and for BN_FOLD publishing the running
statistics as mean / invstd.  Also: the default training / eval plans are unchanged op for op, and Unet.forward picks the
plan variant of its mode, grad state and input."""
import ctypes as C
import hashlib

import pytest
import torch

import oracle
import denoising_diffusion_deep_fake_b200 as d3
from denoising_diffusion_deep_fake_b200 import _lib
from denoising_diffusion_deep_fake_b200.plan import UnetPlan
import op_interpreter as I


def rel(a, b):
    return ((a.double() - b.double()).norm() / (b.double().norm() + 1e-30)).item()


# ------------------------------------------------------------------ interpreter semantics of the frozen BatchNorm
def _run_bn_fold(p):
    I.run_bn_fold(p)
    if p.mean:
        I.view(p.mean, (p.C,)).copy_(I.view(p.running_mean, (p.C,)))
    if p.invstd:
        I.view(p.invstd, (p.C,)).copy_(1.0 / torch.sqrt(I.view(p.running_var, (p.C,)) + p.eps))


def _frozen_apply(p):
    """dx = gamma * invstd * dy' (running statistics: no term from the reductions); dgamma / dbeta from bstats."""
    bs = I.view(p.bstats, (2, p.C), torch.float64)
    if p.dbeta:
        I.view(p.dbeta, (p.C,)).copy_(bs[0].float())
    if p.dgamma:
        I.view(p.dgamma, (p.C,)).copy_(bs[1].float())
    dy = I._masked_dy(p)
    if p.dres:
        I._rows(p.dres, p.count, p.lddres, p.C).copy_(dy)
    I._rows(p.dx, p.count, p.lddx, p.C).copy_(dy * (I.view(p.gamma, (p.C,)) * I.view(p.invstd, (p.C,))))


def _run_bn_bwd(p):
    if not p.frozen:
        return I.run_bn_bwd(p)
    I.run_bn_bwd_reduce(p)
    _frozen_apply(p)


def _run_bn_bwd_apply(p):
    if not p.frozen:
        return I.run_bn_bwd_apply(p)
    _frozen_apply(p)


@pytest.fixture
def interp(monkeypatch):
    monkeypatch.setitem(I._DISPATCH, _lib.OP_BN_FOLD, _run_bn_fold)
    monkeypatch.setitem(I._DISPATCH, _lib.OP_BN_BWD, _run_bn_bwd)
    monkeypatch.setitem(I._DISPATCH, _lib.OP_BN_BWD_APPLY, _run_bn_bwd_apply)
    return I


# ------------------------------------------------------------------ helpers
def make_pair(seed=0, warm_stats=True):
    """Oracle and d3fk.Unet with equal weights; non-default running statistics from two training-mode forwards."""
    torch.manual_seed(seed)
    ref = oracle.Unet()
    with torch.no_grad():
        for n, p in ref.named_parameters():
            if p.dim() == 1 and "segmentation_head" not in n:
                p.uniform_(0.5, 1.5) if n.endswith("weight") else p.uniform_(-0.3, 0.3)
        if warm_stats:
            ref.train()
            for _ in range(2):
                ref(torch.randn(4, 3, 64, 64))
    m = d3.Unet(precision="fp32")
    m.load_state_dict(ref.state_dict())
    return ref, m


def cpu_plan(m, B, H, W, training, dtype=_lib.F32, **kw):
    m._ensure_grad_arena(torch.device("cpu"))
    return UnetPlan(dict(m.named_parameters()), dict(m.named_buffers()), B, H, W, dtype, "cpu", training,
                    grad_arena=m._grad_arena, grad_offsets=m._grad_offsets, **kw)


def run_forward(plan, x):
    y = torch.empty_like(x)
    I.run_ops(plan.pack_ops)
    for i in plan.in_op_indices:
        _lib.op_params(plan.fwd_ops.array[i]).src = x.data_ptr()
    _lib.op_params(plan.fwd_ops.array[plan.out_op_index]).out_nchw = y.data_ptr()
    I.run_ops(plan.fwd_ops)
    return y


def run_backward(plan, dy, dx=None):
    _lib.op_params(plan.bwd_segments[0].array[plan.dy_op_index]).src = dy.data_ptr()
    if dx is not None:
        _lib.op_params(plan.bwd_segments[-1].array[plan.dx_op_index]).out_nchw = dx.data_ptr()
    for seg in plan.bwd_segments:
        I.run_ops(seg)


def param_grads(m, ref):
    out = {}
    for n, p in ref.named_parameters():
        off = m._grad_offsets[n]
        out[n] = m._grad_arena[off:off + p.numel()].view(p.shape).clone()
    return out


def check_grad_errors(errs):
    """The bounds of test_plan_cpu.test_train_plan_matches_oracle, with x.grad in the set."""
    assert errs["segmentation_head.0.weight"] < 1e-5 and errs["segmentation_head.0.bias"] < 1e-5
    assert max(errs.values()) < 2e-2, max(errs, key=errs.get)
    vals = sorted(errs.values())
    assert vals[len(vals) // 2] < 5e-3


# ------------------------------------------------------------------ default plans are unchanged
def _fields(s):
    out = []
    for name, typ in s._fields_:
        v = getattr(s, name)
        if typ is C.c_void_p:
            continue
        if isinstance(v, C.Structure):
            out.append(_fields(v))
        elif isinstance(v, C.Array):
            if typ._type_ is not C.c_void_p:
                out.append(tuple(v))
        else:
            out.append(v)
    return tuple(out)


def plan_fingerprint(plan):
    """sha256 over every op's kind, lane and non-pointer fields (pack, forward, backward segments, the pack table)."""
    lists = [("pack", [(o.kind, o.lane, _fields(_lib.op_params(o))) for o in plan.pack_ops]),
             ("fwd", [(o.kind, o.lane, _fields(_lib.op_params(o))) for o in plan.fwd_ops])]
    for i, seg in enumerate(plan.bwd_segments or []):
        lists.append((f"bwd{i}", [(o.kind, o.lane, _fields(_lib.op_params(o))) for o in seg]))
    n = len(plan.pack_table) // C.sizeof(_lib.PackParams)
    tab = (_lib.PackParams * n).from_buffer_copy(bytes(plan.pack_table.cpu().numpy()))
    lists.append(("table", [_fields(t) for t in tab]))
    return hashlib.sha256(repr(lists).encode()).hexdigest()


# recorded from the plans of the commit before frozen-BN / input-gradient plans existed (B = 2, 64 x 64, default knobs)
_BASE_FINGERPRINTS = {
    (_lib.F32, True): "307673eec6db38b08ac8b32fc38a5f6e2680d3834c2b5ef017994a44354bc4d0",
    (_lib.F32, False): "7d2d18830703c7dd3dc62616fe9c237412de6fc900efcaa16c10b49ed63c0029",
    (_lib.BF16, True): "3ba25fe5db74cbdff9c16f1b0b2db8fdf96bd8ab45cee447982e1d2066a5ef37",
    (_lib.BF16, False): "fd81467da96a540170e4adeebf06bdcab96a9fb99c407d443f655b942ddd5794",
}


@pytest.mark.parametrize("dtype,training", list(_BASE_FINGERPRINTS))
def test_default_plans_unchanged(dtype, training):
    m = d3.Unet(precision="fp32")
    plan = cpu_plan(m, 2, 64, 64, training, dtype=dtype)
    assert plan_fingerprint(plan) == _BASE_FINGERPRINTS[(dtype, training)]


# ------------------------------------------------------------------ plan structure
@pytest.mark.parametrize("dtype", [_lib.F32, _lib.BF16])
@pytest.mark.parametrize("training", [True, False])
def test_dx_variant_adds_only_the_stem_dgrad(dtype, training):
    m = d3.Unet(precision="fp32")
    base = cpu_plan(m, 2, 64, 64, training, dtype=dtype, frozen=not training)
    plan = cpu_plan(m, 2, 64, 64, training, dtype=dtype, frozen=not training, want_dx=True)
    kinds = lambda ol: [(o.kind, o.lane, _fields(_lib.op_params(o))) for o in ol]
    assert kinds(plan.fwd_ops) == kinds(base.fwd_ops)
    assert [kinds(s) for s in plan.bwd_segments[:-1]] == [kinds(s) for s in base.bwd_segments[:-1]]
    last, last0 = kinds(plan.bwd_segments[-1]), kinds(base.bwd_segments[-1])
    assert last[:-1] == last0 and plan.dx_op_index == len(last0) and base.dx_op_index is None
    p = _lib.op_params(plan.bwd_segments[-1].array[plan.dx_op_index])
    assert plan.bwd_segments[-1].array[plan.dx_op_index].kind == _lib.OP_CONV
    assert (p.mode, p.kh, p.kw, p.stride, p.pad, p.c0, p.Cout, p.Hi, p.Wi, p.Ho, p.Wo) == (1, 7, 7, 2, 3, 64, 3, 32, 32, 64, 64)
    assert not p.out and not p.res and not p.scale and not p.stats
    # the stem's BN backward writes the d_raw the dgrad reads
    bn = [o for o in plan.bwd_segments[-1] if o.kind in (_lib.OP_BN_BWD, _lib.OP_BN_BWD_APPLY)][-1]
    assert _lib.op_params(bn).dx == p.src0 and p.w == plan.w_dgrad["encoder.conv1"].data_ptr()
    # the pack table gains exactly the stem's dgrad operand [3][7][7][64]
    tab = lambda pl: (_lib.PackParams * (len(pl.pack_table) // C.sizeof(_lib.PackParams))).from_buffer_copy(
        bytes(pl.pack_table.numpy()))
    t1, t0 = tab(plan), tab(base)
    assert [_fields(t) for t in t1] == [_fields(t) for t in t0]
    stem1 = [t for t in t1 if t.Cin == 3]
    stem0 = [t for t in t0 if t.Cin == 3]
    assert len(stem1) == 1 and stem1[0].w_dgrad and not stem0[0].w_dgrad
    assert tuple(plan.w_dgrad["encoder.conv1"].shape) == (3, 49 * 64)
    assert sum(1 for t in t1 if t.w_dgrad) == sum(1 for t in t0 if t.w_dgrad) + 1


@pytest.mark.parametrize("dtype", [_lib.F32, _lib.BF16])
def test_frozen_plan_structure(dtype):
    m = d3.Unet(precision="fp32")
    plan = cpu_plan(m, 2, 64, 64, False, dtype=dtype, frozen=True)
    assert plan.frozen and not plan.training and plan.bwd_segments is not None
    convbn = [o for o in plan.fwd_ops if o.kind == _lib.OP_CONV_BN]
    assert len(convbn) == 46
    for o in convbn:
        p = _lib.op_params(o)
        assert not p.conv.stats and not p.bn.stats and not p.barrier
        assert not p.conv.scale and p.bn.scale and p.bn.shift
    assert not any(o.kind == _lib.OP_MEMSET for o in plan.fwd_ops)       # no batch statistics to clear
    bwd = [o for s in plan.bwd_segments for o in s if o.kind in (_lib.OP_BN_BWD, _lib.OP_BN_BWD_APPLY)]
    assert len(bwd) == 46
    for o in bwd:
        p = _lib.op_params(o)
        assert p.frozen == 1 and not p.barrier
    # BN_FOLD of every layer, re-packed once per weight version like the eval plan, publishing mean / invstd
    folds = [_lib.op_params(o) for o in plan.pack_ops if o.kind == _lib.OP_BN_FOLD]
    assert len(folds) == 46 and all(f.mean and f.invstd for f in folds)
    eval_folds = [_lib.op_params(o) for o in cpu_plan(m, 2, 64, 64, False, dtype=dtype).pack_ops if o.kind == _lib.OP_BN_FOLD]
    assert len(eval_folds) == 46 and not any(f.mean or f.invstd for f in eval_folds)
    # backward reads the mean / invstd rows the fold writes (fused dgrad-epilogue reductions included)
    rows = {(f.mean, f.invstd) for f in folds}
    for o in bwd:
        p = _lib.op_params(o)
        assert (p.mean, p.invstd) in rows
    for s in plan.bwd_segments:
        for o in s:
            if o.kind == _lib.OP_CONV and _lib.op_params(o).bw_x:
                assert (_lib.op_params(o).bw_mean, _lib.op_params(o).bw_invstd) in rows


# ------------------------------------------------------------------ numerics through the interpreter
@pytest.mark.parametrize("B,H,W", [(2, 64, 64), (3, 32, 96)])
def test_frozen_plan_matches_oracle_eval(interp, B, H, W):
    ref, m = make_pair()
    buffers0 = {k: v.clone() for k, v in m.state_dict().items()}
    assert any(float(v.abs().max()) > 0 for k, v in buffers0.items() if k.endswith("running_mean"))
    torch.manual_seed(1)
    x = torch.randn(B, 3, H, W)
    dy = torch.randn(B, 3, H, W)
    plan = cpu_plan(m, B, H, W, False, frozen=True, want_dx=True)
    y = run_forward(plan, x)
    ref.eval()
    xr = x.clone().requires_grad_()
    y_ref = ref(xr)
    assert rel(y, y_ref.detach()) < 1e-5
    y_ref.backward(dy)
    dx = torch.full_like(x, float("nan"))
    run_backward(plan, dy, dx)
    errs = {n: rel(g, p.grad) for (n, g), p in zip(param_grads(m, ref).items(), ref.parameters())}
    errs["x.grad"] = rel(dx, xr.grad)
    check_grad_errors(errs)
    for k, v in m.state_dict().items():       # running statistics and num_batches_tracked: bitwise unchanged
        assert torch.equal(v, buffers0[k]), k


@pytest.mark.parametrize("B,H,W", [(2, 64, 64)])
def test_train_plan_input_gradient(interp, B, H, W):
    ref, m = make_pair(warm_stats=False)
    sd0 = {k: v.clone() for k, v in m.state_dict().items()}
    torch.manual_seed(2)
    x = torch.randn(B, 3, H, W)
    dy = torch.randn(B, 3, H, W)
    plan0 = cpu_plan(m, B, H, W, True)
    run_forward(plan0, x)
    run_backward(plan0, dy)
    g0 = {n: m._grad_arena[m._grad_offsets[n]:m._grad_offsets[n] + p.numel()].clone() for n, p in m.named_parameters()}
    m.load_state_dict(sd0)                   # the running statistics the first forward moved
    plan = cpu_plan(m, B, H, W, True, want_dx=True)
    run_forward(plan, x)
    dx = torch.full_like(x, float("nan"))
    run_backward(plan, dy, dx)
    for n, p in m.named_parameters():        # parameter gradients equal those of the default plan
        assert torch.equal(m._grad_arena[m._grad_offsets[n]:m._grad_offsets[n] + p.numel()], g0[n]), n
    ref.train()
    xr = x.clone().requires_grad_()
    ref(xr).backward(dy)
    assert rel(dx, xr.grad) < 2e-2


# ------------------------------------------------------------------ Unet.forward: which plan, which autograd
class _StubPlan:
    def __init__(self, B, H, W, frozen, want_dx):
        self.B, self.H, self.W, self.frozen, self.want_dx = B, H, W, frozen, want_dx
        self.generation = 0
        self.pending_backward = False


@pytest.fixture
def stubbed():
    m = d3.Unet(precision="fp32")
    calls = []

    def acquire(x, training, frozen=False, want_dx=False):
        calls.append((training, frozen, want_dx))
        return _StubPlan(x.shape[0], x.shape[2], x.shape[3], frozen and not training, want_dx)

    def run_backward(plan, dy, dx=None):
        calls.append(("bwd", dx is not None))
        if dx is not None:
            dx.fill_(2.0)

    m.__dict__["_acquire_plan"] = acquire
    m.__dict__["_run_forward"] = lambda plan, x: torch.zeros_like(x)
    m.__dict__["_run_backward"] = run_backward
    m.flat_grads = True                      # parameter gradients live in the arena: nothing to slice here
    return m, calls


def test_forward_path_selection(stubbed):
    m, calls = stubbed
    x = torch.randn(1, 3, 32, 32)
    cases = []
    for training in (True, False):
        m.train(training)
        for p in m.parameters():
            p.requires_grad_(True)
        with torch.no_grad():
            cases.append((m(x).grad_fn is None, calls.pop()))
        cases.append((m(x).grad_fn is None, calls.pop()))
        cases.append((m(x.clone().requires_grad_()).grad_fn is None, calls.pop()))
        for p in m.parameters():
            p.requires_grad_(False)
        cases.append((m(x).grad_fn is None, calls.pop()))
        cases.append((m(x.clone().requires_grad_()).grad_fn is None, calls.pop()))
    assert cases == [
        (True, (True, False, False)), (False, (True, False, False)), (False, (True, False, True)),
        (True, (True, False, False)), (False, (True, False, True)),
        (True, (False, False, False)), (False, (False, True, False)), (False, (False, True, True)),
        (True, (False, False, False)), (False, (False, True, True)),
    ]


def test_input_gradient_autograd_contract(stubbed):
    m, calls = stubbed
    for p in m.parameters():
        p.requires_grad_(False)
    for training in (True, False):
        m.train(training)
        x = torch.randn(2, 3, 32, 32, requires_grad=True)
        (g,) = torch.autograd.grad(m(x).sum(), x)
        assert calls[-1] == ("bwd", True) and torch.equal(g, torch.full_like(x, 2.0))
        m(x).sum().backward()
        m(x).sum().backward()
        assert torch.equal(x.grad, torch.full_like(x, 4.0))          # accumulates over two backward calls
        (g,) = torch.autograd.grad(m(x).sum(), x, create_graph=True)
        with pytest.raises(RuntimeError):
            g.sum().backward()                                          # once_differentiable: no silent double backward


def test_eval_backward_refuses_data_parallel(stubbed):
    m, calls = stubbed
    m.eval()
    m.__dict__["_dp_hook"] = lambda i, plan: None
    y = m(torch.randn(1, 3, 32, 32))
    with pytest.raises(NotImplementedError):
        y.sum().backward()
