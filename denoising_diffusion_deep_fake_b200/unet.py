"""Drop-in replacement for the reference denoiser `segmentation_models_pytorch.Unet("resnet34",
encoder_weights=None, in_channels=3, classes=3, activation=None)` built at
d3f/train_denoiser/lit_module.py:41-53 and d3f/train_deep_fake/lit_module.py:49-60.

Same constructor intent, same `forward(x: float32[B,3,H,W]) -> float32[B,3,H,W]`, same parameter /
buffer names (SURVEY Appendix A3) so Lightning checkpoints, `torch.optim.Adam(model.parameters())`,
`copy.deepcopy` (ema_pytorch) and `.train()/.eval()` keep working.  The arithmetic runs in libd3fk
(hand-written sm_100a CUDA behind a C ABI); there is no PyTorch/CPU fallback — calling the module
without the library or off a B200 raises.

Autograd follows nn.Module: a forward with grad enabled and a parameter or the input requiring grad records a graph in BOTH
modes.  Training mode runs the training plan (batch statistics, running-statistics update); eval mode runs the frozen-BN plan
(BatchNorm on its running statistics, which nothing updates) — so an eval-mode forward with grad enabled now records a graph
where it used to return a detached tensor.  Inference callers (the sampler, swap_face, predict_fake, the CLI) run under
torch.no_grad() and take the fused eval plan as before.  `x.requires_grad` adds the input gradient to the backward.
"""
import math

import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import _lib
from .plan import UnetPlan, backward_param_order

_MAX_PLANS_PER_KEY = 4


class _BasicBlock(nn.Module):
    """Parameter holder with torchvision BasicBlock's attribute names (resnet.py:59-87)."""

    def __init__(self, cin, cout, stride):
        super().__init__()
        self.conv1 = nn.Conv2d(cin, cout, 3, stride, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(cout)
        self.conv2 = nn.Conv2d(cout, cout, 3, 1, 1, bias=False)
        self.bn2 = nn.BatchNorm2d(cout)
        self.downsample = None
        if stride != 1 or cin != cout:
            self.downsample = nn.Sequential(nn.Conv2d(cin, cout, 1, stride, bias=False), nn.BatchNorm2d(cout))


class _Encoder(nn.Module):
    def __init__(self):
        super().__init__()
        self.conv1 = nn.Conv2d(3, 64, 7, 2, 3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        cin = 64
        for li, (cout, n) in enumerate(((64, 3), (128, 4), (256, 6), (512, 3)), start=1):
            blocks = []
            for bi in range(n):
                blocks.append(_BasicBlock(cin, cout, 2 if (bi == 0 and li > 1) else 1))
                cin = cout
            setattr(self, f"layer{li}", nn.Sequential(*blocks))
        # torchvision ResNet init (resnet.py:208-213)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)


class _DecoderBlock(nn.Module):
    def __init__(self, cin, cskip, cout):
        super().__init__()
        self.conv1 = nn.Sequential(nn.Conv2d(cin + cskip, cout, 3, padding=1, bias=False), nn.BatchNorm2d(cout),
                                   nn.ReLU(inplace=True))
        self.conv2 = nn.Sequential(nn.Conv2d(cout, cout, 3, padding=1, bias=False), nn.BatchNorm2d(cout),
                                   nn.ReLU(inplace=True))


class _Decoder(nn.Module):
    def __init__(self):
        super().__init__()
        self.blocks = nn.ModuleList(_DecoderBlock(*a) for a in
                                    ((512, 256, 256), (256, 128, 128), (128, 64, 64), (64, 64, 32), (32, 0, 16)))
        for m in self.modules():   # smp initialize_decoder
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_uniform_(m.weight, mode="fan_in", nonlinearity="relu")
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)


class _UnetFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, module, *params):
        want_dx = ctx.needs_input_grad[0]
        plan = module._acquire_plan(x, training=module.training, frozen=not module.training, want_dx=want_dx)
        y = module._run_forward(plan, x)
        ctx.plan, ctx.module = plan, module
        ctx.generation = plan.generation
        ctx.names = module._param_names
        plan.pending_backward = True
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        plan, module = ctx.plan, ctx.module
        if plan.generation != ctx.generation:
            raise RuntimeError("d3fk.Unet: the activations of this forward were overwritten by a later forward "
                               "through the same plan before backward() ran")
        if plan.frozen and module._dp_hook is not None:
            raise NotImplementedError("d3fk.Unet: eval-mode (frozen BatchNorm) backward does not run the data-parallel "
                                      "gradient allreduce; use training mode or disable data parallel")
        dx = None
        if plan.want_dx and ctx.needs_input_grad[0]:
            dx = torch.empty((plan.B, 3, plan.H, plan.W), dtype=torch.float32, device=dy.device)
        module._run_backward(plan, dy, dx)
        plan.pending_backward = False
        if module.flat_grads:
            return (dx, None) + tuple(None for _ in ctx.names)
        flat = module._grad_arena.clone()
        grads = []
        for i, n in enumerate(ctx.names):
            if not ctx.needs_input_grad[2 + i]:
                grads.append(None)
                continue
            off = module._grad_offsets[n]
            p = module._param_dict[n]
            grads.append(flat[off:off + p.numel()].view(p.shape))
        return (dx, None) + tuple(grads)


class Unet(nn.Module):
    """B200-native resnet34 U-Net.  `precision` is "bf16" (tcgen05 tensor cores, fp32 accumulate and fp32
    master weights) or "fp32" (CUDA-core parity mode, 1e-5 vs the oracle)."""

    def __init__(self, encoder_name="resnet34", encoder_weights=None, in_channels=3, classes=3, activation=None,
                 precision="bf16"):
        super().__init__()
        if encoder_name != "resnet34":
            raise ValueError(f"d3fk.Unet implements the encoder the reference configs name ('resnet34'), "
                             f"got {encoder_name!r}")
        if encoder_weights is not None or in_channels != 3 or classes != 3 or activation is not None:
            raise ValueError("d3fk.Unet supports encoder_weights=None, in_channels=3, classes=3, activation=None "
                             "(the only configuration the reference constructs)")
        self.encoder = _Encoder()
        self.decoder = _Decoder()
        self.segmentation_head = nn.Sequential(nn.Conv2d(16, classes, 3, padding=1))
        nn.init.xavier_uniform_(self.segmentation_head[0].weight)
        nn.init.constant_(self.segmentation_head[0].bias, 0)
        self.precision = precision
        self.flat_grads = False
        self._reset_runtime()

    # -------------------------------------------------------------- runtime state (never pickled / copied)
    def _reset_runtime(self):
        self.__dict__["_plans"] = {}
        self.__dict__["_grad_arena"] = None
        self.__dict__["_grad_offsets"] = None
        self.__dict__["_param_dict"] = None
        self.__dict__["_param_names"] = None
        self.__dict__["_packed_version"] = {}
        self.__dict__["_dp_hook"] = None
        self.__dict__["_version_tensors"] = None

    def __deepcopy__(self, memo):
        new = Unet(precision=self.precision)
        new.load_state_dict(self.state_dict())
        dev = next(self.parameters()).device
        new.to(dev)
        for p_new, p_old in zip(new.parameters(), self.parameters()):
            p_new.requires_grad_(p_old.requires_grad)
        new.train(self.training)
        new.flat_grads = False
        return new

    def __getstate__(self):
        state = self.__dict__.copy()
        for k in ("_plans", "_grad_arena", "_grad_offsets", "_param_dict", "_param_names", "_packed_version",
                  "_dp_hook", "_version_tensors"):
            state.pop(k, None)
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)
        self._reset_runtime()

    def _apply(self, fn, *a, **k):
        r = super()._apply(fn, *a, **k)
        self._reset_runtime()
        return r

    @property
    def dtype_code(self):
        if self.precision == "bf16":
            return _lib.BF16
        if self.precision == "fp32":
            return _lib.F32
        raise ValueError(f"precision must be 'bf16' or 'fp32', got {self.precision!r}")

    # -------------------------------------------------------------- plans
    def _ensure_param_tables(self):
        if self._param_dict is None:
            self.__dict__["_param_dict"] = dict(self.named_parameters())
            order = backward_param_order()
            assert set(order) == set(self._param_dict), "parameter naming drifted from the smp scheme"
            self.__dict__["_param_names"] = order
            offs, off = {}, 0
            for n in order:
                offs[n] = off
                off += (self._param_dict[n].numel() + 3) // 4 * 4    # keep every slice 16-byte aligned
            self.__dict__["_grad_offsets"] = offs
            self.__dict__["_grad_numel"] = off

    def _ensure_grad_arena(self, device):
        self._ensure_param_tables()
        if self._grad_arena is None or self._grad_arena.device != device:
            self.__dict__["_grad_arena"] = torch.zeros(self._grad_numel, dtype=torch.float32, device=device)
            if self.flat_grads:
                self.bind_flat_grads()

    def grad_buckets(self):
        """[(start, end)] element ranges of the flat gradient arena completed by backward segment i."""
        self._ensure_param_tables()
        offs = self._grad_offsets
        stage_first = ["segmentation_head.0.weight", "encoder.layer4.2.conv2.weight", "encoder.layer3.5.conv2.weight",
                       "encoder.layer2.3.conv2.weight", "encoder.layer1.2.conv2.weight"]
        starts = [offs[n] for n in stage_first] + [self._grad_numel]
        return [(starts[i], starts[i + 1]) for i in range(len(starts) - 1)]

    def bind_flat_grads(self):
        """Make every parameter's .grad a view of the flat gradient arena (fast trainer path: backward writes
        gradients in place, no per-parameter copies; used with the fused Adam and the bucketed allreduce)."""
        self.flat_grads = True
        dev = next(self.parameters()).device
        self._ensure_param_tables()
        if self._grad_arena is None:
            self.__dict__["_grad_arena"] = torch.zeros(self._grad_numel, dtype=torch.float32, device=dev)
        for n, p in self._param_dict.items():
            off = self._grad_offsets[n]
            p.grad = self._grad_arena[off:off + p.numel()].view(p.shape)

    def _acquire_plan(self, x, training, frozen=False, want_dx=False):
        """The cached plan for x's shape and the variant: training, eval (fused, forward only) or, with training=False and
        frozen=True, the frozen-BN plan; want_dx adds the input gradient to a plan with a backward."""
        if x.dim() != 4 or x.shape[1] != 3:
            raise RuntimeError(f"expected input [B,3,H,W], got {tuple(x.shape)}")
        if x.dtype != torch.float32:
            raise RuntimeError(f"expected float32 input (the reference feeds float32), got {x.dtype}")
        if not x.is_cuda:
            raise _lib.D3fkError("d3fk.Unet runs only on a B200 (sm_100a) CUDA device; there is no CPU path")
        dev = x.device
        _lib.init(dev.index if dev.index is not None else torch.cuda.current_device())
        B, _, H, W = x.shape
        if H % 32 != 0 or W % 32 != 0:
            raise RuntimeError(f"Wrong input shape height={H}, width={W}. Expected image height and width "
                               f"divisible by 32.")
        frozen = bool(frozen) and not training
        want_dx = bool(want_dx) and (training or frozen)
        variant = "train" if training else ("frozen" if frozen else "eval")
        key = (B, H, W, self.dtype_code, variant, want_dx, dev)
        plans = self._plans.setdefault(key, [])
        plans[:] = [p for p in plans if not p.params_moved()]
        for p in plans:
            if not p.pending_backward:
                return p
        if len(plans) >= _MAX_PLANS_PER_KEY:
            p = plans[0]
            p.generation += 1
            p.pending_backward = False
            return p
        params = dict(self.named_parameters())
        buffers = dict(self.named_buffers())
        for n, t in list(params.items()) + list(buffers.items()):
            if t.device != dev:
                raise RuntimeError(f"parameter {n} is on {t.device}, input on {dev}")
        if training or frozen:
            self._ensure_grad_arena(dev)
        plan = UnetPlan(params, buffers, B, H, W, self.dtype_code, dev, training,
                        grad_arena=self._grad_arena, grad_offsets=self._grad_offsets, frozen=frozen, want_dx=want_dx)
        plans.append(plan)
        return plan

    def _new_plan(self, x, training=False):
        """A private plan instance (not cached per shape): the sampler owns one per chain."""
        dev = x.device
        _lib.init(dev.index if dev.index is not None else torch.cuda.current_device())
        B, _, H, W = x.shape
        if training:
            self._ensure_grad_arena(dev)
        return UnetPlan(dict(self.named_parameters()), dict(self.named_buffers()), B, H, W, self.dtype_code, dev, training,
                        grad_arena=self._grad_arena if training else None,
                        grad_offsets=self._grad_offsets if training else None)

    def _weights_version(self):
        ts = self.__dict__.get("_version_tensors")
        if ts is None:      # cached flat list (reset with the other runtime state): this runs twice per training step
            ts = self.__dict__["_version_tensors"] = list(self.parameters()) + list(self.buffers())
        return sum(t._version for t in ts) + self.__dict__.get("_stat_updates", 0)

    def _run_forward(self, plan, x):
        x = x.contiguous()
        stream = torch.cuda.current_stream(x.device).cuda_stream
        if plan.training:
            # master weights change every optimiser step; a trainer that re-packed bucket by bucket right after its Adam
            # update (train.StepOverlap) recorded the version it packed
            if plan.prepacked_version is None or plan.prepacked_version != self._weights_version():
                plan.run_pack(stream)
            plan.prepacked_version = None
            # the kernels update the BN running statistics in place, invisible to tensor._version
            self.__dict__["_stat_updates"] = self.__dict__.get("_stat_updates", 0) + 1
        else:
            ver = self._weights_version()
            if self._packed_version.get(id(plan)) != ver:
                plan.run_pack(stream)      # pack bf16 weights + fold BN once per weight version
                self._packed_version[id(plan)] = ver
        plan.generation += 1
        y = torch.empty_like(x)
        plan.run_forward(x, y, stream)
        return y

    def _run_backward(self, plan, dy, dx=None):
        dy = dy.contiguous()
        stream = torch.cuda.current_stream(dy.device).cuda_stream
        hook = self._dp_hook
        plan.run_backward(dy, stream, after_segment=(lambda i: hook(i, plan)) if hook is not None else None, dx=dx)

    # -------------------------------------------------------------- nn.Module API
    def forward(self, x):
        """Training mode: batch statistics (running statistics updated).  Eval mode: running statistics.  With grad enabled and
        a parameter or `x` requiring grad, the call records a graph in either mode (eval mode: the frozen-BN plan; nothing
        updates the BN buffers); otherwise it runs the plan without autograd (eval mode: the fused eval plan)."""
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            self._ensure_param_tables()
            params = [self._param_dict[n] for n in self._param_names]
            return _UnetFunction.apply(x, self, *params)
        plan = self._acquire_plan(x, training=self.training)
        return self._run_forward(plan, x)
