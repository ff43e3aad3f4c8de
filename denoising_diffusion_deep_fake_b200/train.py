"""Training steps of the reference, re-hosted on the d3fk hot path (plain loop instead of Lightning).

DenoiserModule mirrors d3f/train_denoiser/lit_module.py (training_step :107-126, noising :128-153,
Adam + per-epoch cosine LR :92-100); DeepFakeModule mirrors d3f/train_deep_fake/lit_module.py
(two models + EMA copies, `denoise` and `swap` modes :142-206, two Adam optimisers :113-125).
Data-parallel training (new; the reference is single-GPU) follows PL-DDP semantics: per-rank BN
statistics, mean-reduced gradients — one NCCL allreduce per backward segment, launched on a side
stream as soon as that segment's gradients are final so it overlaps the rest of backward."""
import copy
import math
import os

import torch
import torch.nn as nn

from . import _lib
from .functional import adam_scalars, adam_step_, affine_q_sample, q_sample, random_affine_inverse_maps
from .parallel import allreduce_bucket_
from .loss import MseStructuralSimilarityLoss
from .unet import Unet


class FlatAdam:
    """torch.optim.Adam semantics (eps outside the sqrt, no weight decay) as ONE fused kernel over the
    model's flat parameter / gradient arenas; optional fused EMA lerp target."""

    def __init__(self, model, lr, betas=(0.9, 0.999), eps=1e-8):
        self.model = model
        self.lr, self.betas, self.eps = lr, betas, eps
        self.base_lr = lr
        self.step_count = 0
        dev = next(model.parameters()).device
        model._ensure_grad_arena(dev)
        n = model._grad_numel
        self.flat_p = torch.zeros(n, dtype=torch.float32, device=dev)
        for name, p in model._param_dict.items():
            off = model._grad_offsets[name]
            self.flat_p[off:off + p.numel()].copy_(p.data.reshape(-1))
            p.data = self.flat_p[off:off + p.numel()].view(p.shape)
        model.bind_flat_grads()
        self.m = torch.zeros_like(self.flat_p)
        self.v = torch.zeros_like(self.flat_p)
        # per-step scalars (lr, bias corrections, EMA decay) in device memory, so that the Adam launches can be recorded
        # once in a CUDA graph: dyn_host (pinned) is filled by push_scalars() and copied on the stream before the step
        self.dyn = None

    def enable_device_scalars(self):
        if self.dyn is None:
            self.dyn = torch.zeros(4, dtype=torch.float32, device=self.flat_p.device)
        return self.dyn

    def push_scalars(self, step, ema_decay=0.0):
        """Write the scalars of optimiser step `step` to the device: one tiny launch on the current stream that carries
        the four floats BY VALUE (a host staging buffer could be overwritten before a queued copy has read it — the host
        runs many replayed steps ahead of the device)."""
        vals = adam_scalars(self.lr, self.betas[0], self.betas[1], step, ema_decay)
        op = _lib.make_op(_lib.OP_SET_SCALARS, dst=self.dyn.data_ptr(), v=list(vals))
        _lib.run_single(op, torch.cuda.current_stream(self.dyn.device).cuda_stream)

    def check_aliasing(self):
        name = self.model._param_names[0]
        p = self.model._param_dict[name]
        if p.data_ptr() != self.flat_p.data_ptr() + 4 * self.model._grad_offsets[name]:
            raise RuntimeError("model parameters were re-allocated (.to()/.cuda()) after FlatAdam was built")

    def step(self, ema_flat=None, ema_decay=0.0, grad_scale=1.0):
        """One fused launch over the whole arena.  ema_flat (same layout as flat_p): the kernel's EMA arm also performs
        ema += (1 - ema_decay) * (p_new - ema) in the same pass (ema_pytorch's lerp on the parameters)."""
        self.check_aliasing()
        self.step_count += 1
        if self.dyn is not None:
            self.push_scalars(self.step_count, ema_decay)
        adam_step_(self.flat_p, self.model._grad_arena, self.m, self.v, self.lr, self.betas[0], self.betas[1],
                   self.eps, self.step_count, ema=ema_flat, ema_decay=ema_decay, grad_scale=grad_scale, dyn=self.dyn)
        self.model.__dict__["_stat_updates"] = self.model.__dict__.get("_stat_updates", 0) + 1

    # ---- bucket-wise form of step() (StepOverlap): begin_step, step_range per bucket, end_step
    def begin_step(self, ema_flat=None, ema_decay=0.0):
        self.check_aliasing()
        self.step_count += 1
        self._ema_flat, self._ema_decay = ema_flat, ema_decay
        if self.dyn is not None and not torch.cuda.is_current_stream_capturing():
            self.push_scalars(self.step_count, ema_decay)     # (a graph replay pushes them itself, before the replay)

    def step_range(self, start, end):
        ema = getattr(self, "_ema_flat", None)
        adam_step_(self.flat_p[start:end], self.model._grad_arena[start:end], self.m[start:end], self.v[start:end],
                   self.lr, self.betas[0], self.betas[1], self.eps, self.step_count,
                   ema=None if ema is None else ema[start:end], ema_decay=getattr(self, "_ema_decay", 0.0), dyn=self.dyn)

    def end_step(self, plan=None):
        m = self.model
        m.__dict__["_stat_updates"] = m.__dict__.get("_stat_updates", 0) + 1
        self._ema_flat = None
        if plan is not None:        # the plan's packed operands already hold the updated weights
            plan.prepacked_version = m._weights_version()

    def state_dict(self):
        return {"m": self.m, "v": self.v, "step": self.step_count, "lr": self.lr}

    def load_state_dict(self, sd):
        self.m.copy_(sd["m"]), self.v.copy_(sd["v"])
        self.step_count, self.lr = sd["step"], sd["lr"]


def set_lr(optimizer, lr):
    """Per-epoch cosine LR for either optimiser form (FlatAdam or torch.optim.Adam)."""
    if isinstance(optimizer, FlatAdam):
        optimizer.lr = lr
    else:
        for g in optimizer.param_groups:
            g["lr"] = lr


def cosine_lr(base_lr, epoch, t_max):
    """torch CosineAnnealingLR closed form (eta_min = 0)."""
    return base_lr * (1 + math.cos(math.pi * epoch / t_max)) / 2


class StepOverlap:
    """Everything that FOLLOWS a backward segment, taken off the critical path.  When backward segment i has been
    enqueued, the update stream (ordered behind the main stream and behind libd3fk's weight-gradient streams) runs, for
    gradient bucket i only:  [NCCL mean-allreduce]  ->  [fused Adam]  ->  [re-pack of the bucket's bf16 operands]
    while the main stream goes on with segment i+1 — the deep segments are latency-bound, so these bandwidth-bound
    passes ride along for free.  `finish()` orders the main stream behind the update stream.

    allreduce: a process group is given (data parallel).  adam: a FlatAdam is given (otherwise the caller steps its own
    optimiser after finish())."""

    def __init__(self, model, optimizer=None, group=None, distributed=False):
        self.model, self.optimizer, self.group, self.distributed = model, optimizer, group, distributed
        if distributed:
            import torch.distributed as dist
            self.world = dist.get_world_size(group)
        dev = next(model.parameters()).device
        self.comm = torch.cuda.Stream(dev)
        self.buckets = model.grad_buckets()
        self.armed = False          # the optimiser part runs only inside a training step that asked for it
        self.ema_target = (None, 0.0)   # (flat EMA arena, decay) the Adam launches of THIS step also lerp (swap mode)
        self.stepped = False
        self._plan = None
        model.__dict__["_dp_hook"] = self.after_segment

    def after_segment(self, i, plan=None):
        do_adam = self.armed and self.optimizer is not None
        if not (self.distributed or do_adam):
            return
        cur = torch.cuda.current_stream()
        ev = torch.cuda.Event()
        ev.record(cur)
        self.comm.wait_event(ev)                           # BN / bias gradients, dgrad reads of the packed weights: main stream
        _lib.side_stream_join(self.comm.cuda_stream)       # weight gradients: libd3fk's side streams
        s, e = self.buckets[i]
        with torch.cuda.stream(self.comm):
            if self.distributed:
                allreduce_bucket_(self.model._grad_arena, s, e, self.group)
            if do_adam:
                if i == 0:
                    self.optimizer.begin_step(*self.ema_target)
                self.optimizer.step_range(s, e)
                if plan is not None:
                    plan.run_pack_bucket(i, self.comm.cuda_stream)
                    self._plan = plan
                if i == len(self.buckets) - 1:
                    self.stepped = True

    def wait(self):
        torch.cuda.current_stream().wait_stream(self.comm)

    def finish(self):
        """Main stream waits for the update stream; returns True when the optimiser step (and the re-pack) already ran."""
        self.wait()
        stepped, self.stepped = self.stepped, False
        if stepped:
            self.optimizer.end_step(self._plan)
        self._plan = None
        return stepped


GradAllReduce = StepOverlap    # the allreduce-only use (optimizer=None) keeps its old name


class GraphedStep:
    """The training step behind the noising — U-Net forward, criterion, backward with its weight-gradient side streams,
    per-bucket [allreduce ->] Adam -> re-pack on the update stream — recorded ONCE as a CUDA graph and replayed per step
    (SURVEY §7 step 7).  The step is static: every buffer belongs to the plan or to the graph's private pool, the kernels'
    programmatic-dependent-launch edges are kept by the capture, and what changes from step to step lives in device memory
    (Adam's lr / bias corrections: FlatAdam.dyn; BN's num_batches_tracked; the Philox offset stays outside: the noising
    launch is issued eagerly in front of the replay and writes into the graph's static input).

    One graph per input buffer address (a caller that reuses its device buffers — bench.py, a double-buffered loader —
    replays directly; any other batch is copied into a module-owned static buffer first).  A graph is dropped whenever the
    weights were changed from outside (load_state_dict, manual edits), which the version counter reveals."""

    MAX_POINTER_GRAPHS = 4

    def __init__(self, module):
        self.module = module
        self.entries = {}       # key -> dict(graph, x, noisy, loss, version)
        self.seen = {}          # data_ptr -> times seen (pointer graphs are built for repeat customers only)
        self.static_x = {}      # shape -> module-owned input buffer
        self.eager_steps = 0    # eager steps since the last invalidation: capture needs warmed plans and a valid pre-pack
        self.replays = 0
        self.kernels_replayed = 0   # libd3fk kernel nodes executed through replays (the library's own counter sees only
                                    # the launches of the capture)

    def invalidate(self):
        self.entries.clear()
        self.eager_steps = 0

    def _capture(self, x):
        mod = self.module
        model, opt = mod.model, mod.optimizer
        noisy = torch.empty_like(x)
        plan = model._acquire_plan(noisy, training=True)
        if plan.prepacked_version is None or plan.prepacked_version != model._weights_version():
            return None                      # the forward would start with a full pack: not the steady state yet
        host = (opt.step_count, model.__dict__.get("_stat_updates", 0), plan.generation, plan.prepacked_version)
        g = torch.cuda.CUDAGraph()
        k0 = _lib.launch_count()
        with torch.cuda.graph(g):
            loss = mod._step_body(x, noisy)
        kernels = _lib.launch_count() - k0
        # nothing ran during the capture: take back the host-side bookkeeping it advanced
        opt.step_count, model.__dict__["_stat_updates"], plan.generation, plan.prepacked_version = host
        plan.pending_backward = False
        return dict(graph=g, x=x, noisy=noisy, loss=loss, plan=plan, kernels=kernels)

    def step(self, image, noise=None, y=None):
        """Returns the loss tensor, or None when the step has to run eagerly (warm-up, stale graph)."""
        mod = self.module
        model, opt = mod.model, mod.optimizer
        if self.eager_steps < 2:
            self.eager_steps += 1
            return None
        ptr = image.data_ptr()
        key = (ptr, tuple(image.shape))
        ent = self.entries.get(key)
        if ent is None:
            self.seen[ptr] = self.seen.get(ptr, 0) + 1
            n_ptr = sum(1 for k in self.entries if k[0] != "static")
            if self.seen[ptr] >= 2 and n_ptr < self.MAX_POINTER_GRAPHS and image.is_contiguous():
                ent = self._capture(image)
                if ent is None:
                    return None
                self.entries[key] = ent
            else:
                key = ("static", tuple(image.shape))
                ent = self.entries.get(key)
                if ent is None:
                    ent = self._capture(torch.empty_like(image, memory_format=torch.contiguous_format))
                    if ent is None:
                        return None
                    self.entries[key] = ent
        if ent["plan"].prepacked_version != model._weights_version() or ent["plan"].params_moved():
            self.invalidate()                # weights were touched from outside: eager steps re-establish the steady state
            return None
        if ent["x"].data_ptr() != ptr:
            ent["x"].copy_(image)
        mod._noise_into(ent["x"], ent["noisy"], noise, y)
        opt.push_scalars(opt.step_count + 1)
        ent["graph"].replay()
        # the host-side bookkeeping of the step the replay just enqueued
        opt.step_count += 1
        model.__dict__["_stat_updates"] = model.__dict__.get("_stat_updates", 0) + 2      # BN running stats + Adam
        ent["plan"].generation += 1
        ent["plan"].prepacked_version = model._weights_version()
        self.replays += 1
        self.kernels_replayed += ent["kernels"]
        return ent["loss"]


class DenoiserModule(nn.Module):
    """train_denoiser LitModule, minus Lightning.  hparams: encoder_name, learning_rate,
    noise_exponential_sampling_lambda, cosine_scheduler_max_epoch (+ precision, seed: new)."""

    def __init__(self, **hparams):
        super().__init__()
        self.hparams = dict(hparams)
        p = self.hparams
        self.model = Unet(encoder_name=p["encoder_name"], encoder_weights=None, in_channels=3, classes=3,
                          activation=None, precision=p.get("precision", "bf16"))
        self.training_criterion = MseStructuralSimilarityLoss(-1.0, 1.0)
        self.global_step = 0
        self.current_epoch = 0
        self.optimizer = None
        self.allreduce = None
        self._aug_generator = None
        self._graphed = None       # GraphedStep once the fused trainer is in its steady state (False: disabled)

    def forward(self, image):
        return self.model(image)

    def configure_optimizers(self, fused=True, overlap=True):
        """fused: one-kernel Adam over the flat arenas; overlap (fused only): the Adam update and the bf16 re-pack of each
        gradient bucket run on a second stream underneath the rest of backward (StepOverlap)."""
        p = self.hparams
        if fused:
            self.optimizer = FlatAdam(self.model, lr=p["learning_rate"])
            if overlap and os.environ.get("D3FK_OVERLAP_STEP", "1") != "0":
                self.allreduce = StepOverlap(self.model, self.optimizer)
        else:
            self.optimizer = torch.optim.Adam(self.model.parameters(), lr=p["learning_rate"])
        return self.optimizer

    def enable_data_parallel(self, group=None):
        overlap_adam = self.allreduce is not None and self.allreduce.optimizer is not None
        self.allreduce = StepOverlap(self.model, self.optimizer if overlap_adam else None, group, distributed=True)

    def blend_random_amount_of_noise_with_each_sample(self, batch, noise=None, y=None):
        p = self.hparams
        return q_sample(batch, p["noise_exponential_sampling_lambda"], noise=noise, y=y,
                        seed=p.get("seed", 0), offset=self.global_step)

    def augment_and_blend(self, batch, noise=None, y=None):
        """`image = self.shared_augmentation_sequence(image)` + the noising (lit_module.py:55-65, :113-115) as one kernel:
        returns (augmented image = the loss target, noisy augmented image = the network input)."""
        p = self.hparams
        B, _, H, W = batch.shape
        if self._aug_generator is None:
            self._aug_generator = torch.Generator().manual_seed(int(p.get("seed", 0)) + 0x5EED)
        maps = random_affine_inverse_maps(B, H, W, generator=self._aug_generator)
        return affine_q_sample(batch, maps, p["noise_exponential_sampling_lambda"], noise=noise, y=y,
                               seed=p.get("seed", 0), offset=self.global_step)

    def _noise_into(self, image, noisy, noise=None, y=None):
        """The noising launch in front of a graph replay: image -> noisy (both static buffers of the graph)."""
        p = self.hparams
        q_sample(image, p["noise_exponential_sampling_lambda"], noise=noise, y=y, seed=p.get("seed", 0),
                 offset=self.global_step, out=noisy)

    def _step_body(self, image, image_noisy):
        """Forward, criterion, backward and the overlapped per-bucket optimiser work, without autograd objects (the body a
        GraphedStep records)."""
        model, ov = self.model, self.allreduce
        plan = model._acquire_plan(image_noisy, training=True)
        image_prediction = model._run_forward(plan, image_noisy)
        loss, grad = self.training_criterion.value_and_grad(image_prediction, image)
        ov.armed = True
        try:
            model._run_backward(plan, grad)
        finally:
            ov.armed = False
        if not ov.finish():
            raise RuntimeError("the overlapped optimiser step did not run")
        return loss

    def _graph_eligible(self):
        if self._graphed is False:
            return False
        ok = (isinstance(self.optimizer, FlatAdam) and self.allreduce is not None and self.allreduce.optimizer is not None
              and self.model.training and not self.hparams.get("augment", False)
              and self.hparams.get("cuda_graph", os.environ.get("D3FK_TRAIN_GRAPH", "1") != "0")
              and all(p.requires_grad for p in self.model.parameters()))
        if ok and self.allreduce.distributed:
            # the NCCL allreduces of the gradient buckets are captured with the step (every rank captures on the same
            # step); measured at 2 GPUs: 4.33 -> 4.22 ms per step.  D3FK_TRAIN_GRAPH_DP=0 keeps data parallel eager.
            ok = os.environ.get("D3FK_TRAIN_GRAPH_DP", "1") != "0"
        return ok

    def training_step(self, image, noise=None, y=None):
        """[affine augmentation ->] noising -> U-Net -> MSE+SSIM loss -> backward -> Adam (lit_module.py:107-126 + the
        optimiser step Lightning would take).  Returns the loss tensor (no host sync).  hparam `augment` (default False:
        the benchmark feeds pre-augmented tensors) switches the reference's kornia RandomAffine on.
        With the fused optimiser the step is replayed from a CUDA graph after two eager warm-up steps (GraphedStep;
        hparam `cuda_graph: false` or D3FK_TRAIN_GRAPH=0 keeps it eager)."""
        if self._graph_eligible():
            if self._graphed is None:
                self.optimizer.enable_device_scalars()
                self._graphed = GraphedStep(self)
            loss = self._graphed.step(image, noise, y)
            if loss is not None:
                self.global_step += 1
                self._check_device_flag()
                return loss
        if self.hparams.get("augment", False):
            image, image_noisy = self.augment_and_blend(image, noise, y)
        else:
            image_noisy = self.blend_random_amount_of_noise_with_each_sample(image, noise, y)
        image_prediction = self.model(image_noisy)
        # value and dL/dprediction from the one fused launch; the U-Net backward is seeded directly (no autograd node for
        # the criterion, no grad * grad_output pass)
        loss, grad = self.training_criterion.value_and_grad(image_prediction, image)
        if not isinstance(self.optimizer, FlatAdam):
            self.optimizer.zero_grad(set_to_none=True)
        stepped = False
        if self.allreduce is not None:
            self.allreduce.armed = True
            try:
                image_prediction.backward(grad)
            finally:
                self.allreduce.armed = False
            stepped = self.allreduce.finish()
        else:
            image_prediction.backward(grad)
        if not stepped:
            self.optimizer.step()
        self.global_step += 1
        self._check_device_flag()
        return loss

    def _check_device_flag(self, every=512):
        """A kernel watchdog traps (sticky CUDA error) — this additionally polls the device error flag every `every` steps
        (a 4-byte read; it synchronises, hence not every step)."""
        if self.global_step % every == 0 and _lib.load().d3fk_device_error_flag():
            raise _lib.D3fkError("a d3fk kernel reported a barrier watchdog timeout; the results of this run are void")

    def on_epoch_end(self):
        self.current_epoch += 1
        lr = cosine_lr(self.hparams["learning_rate"], self.current_epoch, self.hparams["cosine_scheduler_max_epoch"])
        set_lr(self.optimizer, lr)


class EMA(nn.Module):
    """ema_pytorch.EMA(model, beta, update_every, include_online_model=False) semantics (SURVEY Appendix B2):
    copy for the first `update_after_step` updates, then lerp with decay
    clamp(1-(1+(step-101)/inv_gamma)^-power, 0, beta) over float params and buffers.

    Fast path (`bind_flat`): the EMA parameters become views of ONE flat fp32 arena laid out like the online model's
    FlatAdam arena, and the parameter lerp of the next `update()` is performed by the EMA arm of the fused Adam kernel
    (d3fk_adam) in the same pass that updates the online weights — `planned_lerp()` tells the trainer whether the next
    update() will lerp and with which decay; `update()` then only advances the counters and lerps the (tiny) BN buffers.
    The schedule is driven from host mirrors of the `step` / `initted` buffers (no device sync per step); a
    load_state_dict re-synchronises them (resume)."""

    def __init__(self, model, beta=0.9999, update_after_step=100, update_every=10, inv_gamma=1.0, power=2 / 3,
                 min_value=0.0, include_online_model=True):
        super().__init__()
        self.beta, self.update_after_step, self.update_every = beta, update_after_step, update_every
        self.inv_gamma, self.power, self.min_value = inv_gamma, power, min_value
        if include_online_model:
            self.online_model = model
        else:
            self.online_model = [model]
        self.ema_model = copy.deepcopy(model)
        self.ema_model.requires_grad_(False)
        self.register_buffer("initted", torch.tensor(False))
        self.register_buffer("step", torch.tensor(0))
        self._step_host = 0
        self._initted_host = False
        self._flat = None            # flat arena of the EMA parameters (bind_flat)
        self._online_flat = None     # the online model's FlatAdam arena
        self._preapplied = False     # the parameter lerp of the NEXT update() already ran inside the Adam kernel
        self.register_load_state_dict_post_hook(EMA._resync_host_mirrors)

    @staticmethod
    def _resync_host_mirrors(module, incompatible_keys):
        module._step_host = int(module.step)
        module._initted_host = bool(module.initted)
        module._preapplied = False

    @property
    def model(self):
        return self.online_model if isinstance(self.online_model, nn.Module) else self.online_model[0]

    def get_current_decay(self, step):
        epoch = max(step - self.update_after_step - 1, 0)
        if epoch <= 0:
            return 0.0
        value = 1 - (1 + epoch / self.inv_gamma) ** -self.power
        return min(max(value, self.min_value), self.beta)

    @torch.no_grad()
    def bind_flat(self, optimizer):
        """Re-home the EMA parameters in one flat arena with the layout of `optimizer.flat_p` (a FlatAdam over the online
        model).  Call after the module sits on its device."""
        model, ema = self.model, self.ema_model
        model._ensure_param_tables()
        flat = torch.zeros_like(optimizer.flat_p)
        ema_params = dict(ema.named_parameters())
        for name, off in model._grad_offsets.items():
            p = ema_params[name]
            flat[off:off + p.numel()].copy_(p.data.reshape(-1))
            p.data = flat[off:off + p.numel()].view(p.shape)
        self._flat, self._online_flat = flat, optimizer.flat_p

    def _flat_ok(self):
        """The flat views survive only as long as nobody re-allocated the parameters (.to() / .cuda())."""
        if self._flat is None:
            return False
        name = self.model._param_names[0]
        off = self.model._grad_offsets[name]
        ok = (dict(self.ema_model.named_parameters())[name].data_ptr() == self._flat.data_ptr() + 4 * off
              and self.model._param_dict[name].data_ptr() == self._online_flat.data_ptr() + 4 * off)
        if not ok:
            self._flat = self._online_flat = None
        return ok

    def planned_lerp(self):
        """(flat EMA arena, decay) if the next update() call will lerp the parameters, else None."""
        step = self._step_host
        if step % self.update_every != 0 or step <= self.update_after_step or not self._initted_host:
            return None
        if self._preapplied or not self._flat_ok():
            return None
        return self._flat, self.get_current_decay(step + 1)

    def mark_preapplied(self):
        self._preapplied = True
        self._bump_version()

    def _bump_version(self):
        d = self.ema_model.__dict__
        if "_stat_updates" in d or hasattr(self.ema_model, "_weights_version"):
            d["_stat_updates"] = d.get("_stat_updates", 0) + 1     # in-place writes invisible to tensor._version

    @torch.no_grad()
    def _copy(self):
        if self._flat_ok():
            self._flat.copy_(self._online_flat)
            self._bump_version()
        else:
            for e, m in zip(self.ema_model.parameters(), self.model.parameters()):
                e.copy_(m)
        for e, m in zip(self.ema_model.buffers(), self.model.buffers()):
            e.copy_(m)

    @torch.no_grad()
    def update(self):
        step = self._step_host
        self._step_host += 1
        self.step += 1
        if step % self.update_every != 0:
            return
        if step <= self.update_after_step:
            self._copy()
            return
        if not self._initted_host:
            self._copy()
            self._initted_host = True
            self.initted.fill_(True)
        decay = self.get_current_decay(self._step_host)
        if self._preapplied:
            self._preapplied = False          # parameters: done by the EMA arm of the online model's last Adam launch
        elif self._flat_ok():
            self._flat.lerp_(self._online_flat, 1 - decay)
            self._bump_version()
        else:
            ep = [e for e in self.ema_model.parameters() if e.is_floating_point()]
            mp = [m for e, m in zip(self.ema_model.parameters(), self.model.parameters()) if e.is_floating_point()]
            torch._foreach_lerp_(ep, mp, 1 - decay)
        eb = [e for e in self.ema_model.buffers() if e.is_floating_point()]
        mb = [m for e, m in zip(self.ema_model.buffers(), self.model.buffers()) if e.is_floating_point()]
        if eb:
            torch._foreach_lerp_(eb, mb, 1 - decay)

    def forward(self, *a, **k):
        return self.ema_model(*a, **k)


class DeepFakeModule(nn.Module):
    """train_deep_fake LitModule, minus Lightning: model_a/model_b (+ EMA copies in swap mode)."""

    def __init__(self, **hparams):
        super().__init__()
        self.hparams = dict(hparams)
        p = self.hparams
        prec = p.get("precision", "bf16")
        self.model_a = Unet(encoder_name=p["encoder_name"], precision=prec)
        self.model_b = Unet(encoder_name=p["encoder_name"], precision=prec)
        self.ema_model_a = self.create_ema_model(self.model_a)
        self.ema_model_b = self.create_ema_model(self.model_b)
        self.criterion = MseStructuralSimilarityLoss(-1.0, 1.0)
        self.global_step = 0
        self.current_epoch = 0
        self.logged = {}
        self._aug_generator = None
        self.optimizer_a = self.optimizer_b = None
        self.overlap_a = self.overlap_b = None

    def create_ema_model(self, model):
        p = self.hparams
        if p["mode"] == "swap":
            return EMA(model, beta=p["ema_beta"], update_every=p["ema_update_every"], include_online_model=False)
        return None

    def configure_optimizers(self, fused=None, overlap=True):
        """Two Adams with betas from the config (lit_module.py:113-125).  fused (default: whenever the models sit on a CUDA
        device): one-kernel FlatAdam per model over its flat arenas, the EMA copies re-homed in flat arenas so the Adam
        launch also performs their parameter lerp, and — `overlap` — the per-bucket Adam / re-pack running underneath
        backward (StepOverlap), as in DenoiserModule.  fused=False keeps torch.optim.Adam over .parameters()."""
        p = self.hparams
        betas = (p["adam_b1"], p["adam_b2"])
        if fused is None:
            fused = next(self.model_a.parameters()).is_cuda
        if fused:
            self.optimizer_a = FlatAdam(self.model_a, lr=p["learning_rate"], betas=betas)
            self.optimizer_b = FlatAdam(self.model_b, lr=p["learning_rate"], betas=betas)
            if overlap and os.environ.get("D3FK_OVERLAP_STEP", "1") != "0":
                self.overlap_a = StepOverlap(self.model_a, self.optimizer_a)
                self.overlap_b = StepOverlap(self.model_b, self.optimizer_b)
            if self.ema_model_a is not None:
                self.ema_model_a.bind_flat(self.optimizer_a)
                self.ema_model_b.bind_flat(self.optimizer_b)
        else:
            self.optimizer_a = torch.optim.Adam(self.model_a.parameters(), lr=p["learning_rate"], betas=betas)
            self.optimizer_b = torch.optim.Adam(self.model_b.parameters(), lr=p["learning_rate"], betas=betas)
        return [self.optimizer_a, self.optimizer_b]

    def blend_random_amount_of_noise_with_each_sample(self, batch, noise=None, y=None):
        p = self.hparams
        self._noise_calls = getattr(self, "_noise_calls", 0) + 1
        return q_sample(batch, p["noise_exponential_sampling_lambda"], noise=noise, y=y, seed=p.get("seed", 0),
                        offset=self._noise_calls)

    def augment(self, batch):
        """The reference augments in its DataLoader workers: A.ShiftScaleRotate(shift 0.2, scale 0.1, rotate 15, border 0,
        p=0.7) (lit_module.py:99-111).  Here: the same parameter distribution, applied on the device by the affine kernel
        (bilinear, zero border); samples that draw "no augmentation" get the identity map.  hparam `augment` (default off:
        tensor-level callers and the benchmark feed ready batches) switches it on; the CLI does for list-file data."""
        B, _, H, W = batch.shape
        if self._aug_generator is None:
            self._aug_generator = torch.Generator().manual_seed(int(self.hparams.get("seed", 0)) + 0xA06)
        maps = random_affine_inverse_maps(B, H, W, degrees=15.0, translate=(0.2, 0.2), scale=(0.9, 1.1), p=0.7,
                                          generator=self._aug_generator)
        aug, _ = affine_q_sample(batch, maps, 1.0, fixed_r=0.0)
        return aug

    def training_step(self, batch_a, batch_b, noise=None, y=None):
        """Both optimiser passes of one Lightning batch (lit_module.py:142-156).  noise / y: optional dicts {"a": ..., "b": ...}
        of supplied noising draws (parity runs)."""
        out = {}
        if self.optimizer_a is None:
            self.configure_optimizers()
        if self.hparams.get("augment", False):
            batch_a, batch_b = self.augment(batch_a), self.augment(batch_b)
        for name, real, real_model, fake_model, own_ema, opt, ov in (
                ("a", batch_a, self.model_a, self.ema_model_b, self.ema_model_a, self.optimizer_a, self.overlap_a),
                ("b", batch_b, self.model_b, self.ema_model_a, self.ema_model_b, self.optimizer_b, self.overlap_b)):
            self._draws = (None if noise is None else noise[name], None if y is None else y[name])
            if isinstance(opt, FlatAdam):
                out[name] = self._fused_step_for_one_model(name, real, real_model, fake_model, own_ema, opt, ov)
            else:
                opt.zero_grad(set_to_none=True)
                loss = self.training_step_for_one_model(name, real, real_model, fake_model)
                loss.backward()
                opt.step()
                out[name] = loss
        self._draws = (None, None)
        self.global_step += 1
        return out

    def _fused_step_for_one_model(self, name, real, real_model, fake_model, own_ema, opt, ov):
        """One optimiser pass on the fast path: loss value and dL/dprediction from the one criterion launch, the U-Net
        backward seeded directly, gradients in the flat arena, ONE Adam launch (per bucket, underneath backward, with
        StepOverlap) whose EMA arm also lerps this model's EMA copy when its next update() is a lerp."""
        real_prediction = self._prediction_for_one_model(name, real, real_model, fake_model)
        loss, grad = self.criterion.value_and_grad(real_prediction, real)
        self.logged[f"loss_{self.hparams['mode']}/train_{name}"] = loss
        planned = own_ema.planned_lerp() if own_ema is not None else None
        ema_flat, decay = planned if planned is not None else (None, 0.0)
        stepped = False
        if ov is not None:
            ov.armed, ov.ema_target = True, (ema_flat, decay)
            try:
                real_prediction.backward(grad)
            finally:
                ov.armed = False
            stepped = ov.finish()
        else:
            real_prediction.backward(grad)
        if not stepped:
            opt.step(ema_flat=ema_flat, ema_decay=decay)
        if planned is not None:
            own_ema.mark_preapplied()
        return loss

    def _prediction_for_one_model(self, name, real, real_model, fake_model):
        """The data flow of training_{denoise,swap}_step_for_one_model up to the prediction (lit_module.py:168-197)."""
        noise, y = getattr(self, "_draws", (None, None))
        if self.hparams["mode"] == "denoise":
            with torch.no_grad():
                noisy_real = self.blend_random_amount_of_noise_with_each_sample(real, noise, y)
            return real_model(noisy_real)
        fake_model.update()
        with torch.no_grad():
            fake = fake_model(real)                        # one pass, BN in train mode as in the reference
            self.logged[f"swap_difference/{name}"] = nn.functional.mse_loss(real, fake)
            noisy_fake = self.blend_random_amount_of_noise_with_each_sample(fake, noise, y)
        return real_model(noisy_fake)

    def training_step_for_one_model(self, name, real, real_model, fake_model):
        if self.hparams["mode"] == "denoise":
            return self.training_denoise_step_for_one_model(name, real, real_model)
        return self.training_swap_step_for_one_model(name, real, real_model, fake_model)

    def training_denoise_step_for_one_model(self, name, real, real_model):
        real_prediction = self._prediction_for_one_model(name, real, real_model, None)
        loss = self.criterion(real_prediction, real)
        self.logged[f"loss_denoise/train_{name}"] = loss.detach()
        return loss

    def training_swap_step_for_one_model(self, name, real, real_model, fake_model):
        real_prediction = self._prediction_for_one_model(name, real, real_model, fake_model)
        loss = self.criterion(real_prediction, real)
        self.logged[f"loss_swap/train_{name}"] = loss.detach()
        return loss

    def on_epoch_end(self):
        self.current_epoch += 1
        lr = cosine_lr(self.hparams["learning_rate"], self.current_epoch, self.hparams["cosine_scheduler_max_epoch"])
        for o in (self.optimizer_a, self.optimizer_b):
            set_lr(o, lr)

    @torch.no_grad()
    def predict_fake(self, real, model_a_or_b, mask=None):
        """predict_fake (lit_module.py:251-270).  Two input forms:
        * the reference's: one uint8 BGR frame [H,W,3] (numpy, as cv2 delivers it) or a batch [N,H,W,3] (numpy or a uint8
          CUDA tensor) -> the fake frame(s), same type and layout.  Normalisation, the network and the conversion back
          all run on the device (d3fk_frames_to_tensor / d3fk_tensor_to_frames); model "a" uses mean_b / std_b and
          model "b" mean_a / std_a, as the reference does (:253-257).
        * a normalised fp32 tensor [B,3,H,W] -> the network output (tensor-level use inside training code).
        mask (optional; 1 = swap, 0 = keep the input, fractions feather): the output is m*fake + (1 - m)*input, fused into
        one kernel after the network.  Any form functional.normalize_mask takes; with uint8 frames also a uint8 [H,W] or
        [N,H,W] mask in 0..255 (numpy or torch, as cv2 produces masks), scaled by 1/255.  Where m == 0 the output frame
        is the input's own round trip through normalisation, tensor_to_frames(frames_to_tensor(frame))."""
        import numpy as np
        from .functional import composite_, frames_to_tensor, normalize_mask, tensor_to_frames
        model = self.model_a if model_a_or_b == "a" else self.model_b
        is_numpy = isinstance(real, np.ndarray)
        frames = torch.from_numpy(np.ascontiguousarray(real)) if is_numpy else real
        if isinstance(mask, np.ndarray):
            mask = torch.from_numpy(np.ascontiguousarray(mask))
        if mask is not None and mask.dtype == torch.uint8:
            if frames.dtype != torch.uint8:
                raise TypeError("a uint8 mask goes with uint8 frames; give a float32 or bool mask for a normalised tensor")
            if mask.dim() == 3:
                mask = mask.unsqueeze(1)                 # [N,H,W] -> [N,1,H,W]
            mask = mask.to(torch.float32) / 255.0

        def composited(out, x):
            if mask is None:
                return out
            B, _, H, W = x.shape
            return composite_(out, x, normalize_mask(mask, B, H, W).to(out.device))

        was = model.training
        model.eval()
        try:
            if frames.dtype != torch.uint8:
                return composited(model(frames), frames)
            p = self.hparams
            other = "b" if model_a_or_b == "a" else "a"
            mean, std = p.get(f"mean_{other}", [0.5] * 3), p.get(f"std_{other}", [0.5] * 3)
            single = frames.dim() == 3
            dev = next(model.parameters()).device
            x = frames_to_tensor(frames.to(dev, non_blocking=True), mean, std)
            fake = tensor_to_frames(composited(model(x), x), mean, std)
            fake = fake[0] if single else fake
            return fake.cpu().numpy() if is_numpy else fake
        finally:
            model.train(was)
