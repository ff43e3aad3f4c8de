"""Iterative reverse-diffusion sampler over the x0-predicting U-Net (SURVEY §3.4 / §8a row S).

The reference swaps a face with ONE forward pass (`fake = fake_model(real)`,
d3f/train_deep_fake/lit_module.py:187-189, :259-270); BASELINE.json defines an N-step sampler on the
same network.  Each step = eval-mode U-Net forward (BN folded into the conv epilogues) + one fused
posterior kernel + a device-side step counter, recorded ONCE as a CUDA graph and replayed N times —
the graph is step-independent because the coefficients are read from a device table indexed by the
counter.  `n_steps=1, r_start=0` is the reference-exact single pass.  Batch-sharded across GPUs with no
communication (each rank owns its images, graph and Philox stream).

Chains (opt-in, `chains=` / D3FK_SAMPLER_CHAINS): in eval mode the images of a batch are independent (BatchNorm is a folded
affine), so the batch can be split into sub-batches, each with its own plan, step counter and CUDA stream, captured as
parallel branches of the same graph.  Measured on B200 at B=64 @128x128 this LOSES (1.11 ms/step with one chain, 1.18 with
two, 1.43 with four): the forward is bound by kernel throughput, not by launch latency, and smaller sub-batches only add
per-kernel fixed cost.  It pays only for small batches of large images sharing one GPU; default 1.

Masked sampling (`masked=True`; replacement inpainting, as RePaint without resampling): every step blends the update with
the source noised to the step's target ratio, x = m*post + (1 - m)*known, inside the same posterior kernel — the mask
adds no launch.  At the last step known is the source itself, so where the mask is 0 the result is the source exactly.

Solvers (`solver=`): "posterior" is the first-order update (DDIM at eta 0, DDPM ancestral at eta 1); "dpmpp_2m" is the
second-order multistep DPM-Solver++ 2M, which extrapolates x0_hat with the previous step's (kept in one more [B,3,H,W]
buffer) inside the same fused posterior kernel — no extra forward and no extra launch per step.  Its order shows on a grid
uniform in log-SNR (`schedule="logsnr"`, the default for "dpmpp_2m"); on the linear grid it gains almost nothing."""
import os

import torch

from . import _lib
from ._lib import make_op, op_params
from .functional import (composite_, dpmpp_2m_coef_table, dpmpp_2m_step_, noise_ratio_grid, normalize_mask,
                         posterior_coef_table, posterior_step_, q_sample)

SOLVERS = ("posterior", "dpmpp_2m")
SCHEDULES = ("linear", "logsnr")


class Sampler:
    def __init__(self, model, batch, height, width, n_steps, r_start=1.0, eta=0.0, seed=0, use_graph=True,
                 steps_per_graph=1, chains=None, masked=False, solver="posterior", schedule=None, r_min=1e-3):
        """solver: "posterior" (first order) or "dpmpp_2m" (second-order multistep; see functional.dpmpp_2m_coeffs).
        schedule: the ratio grid, "linear" or "logsnr" (functional.noise_ratio_grid, with r_min); None picks the solver's:
        linear for "posterior", logsnr for "dpmpp_2m"."""
        if solver not in SOLVERS:
            raise ValueError(f"unknown solver {solver!r}: one of {SOLVERS}")
        if schedule is None:
            schedule = "linear" if solver == "posterior" else "logsnr"
        if schedule not in SCHEDULES:
            raise ValueError(f"unknown schedule {schedule!r}: one of {SCHEDULES}")
        p = next(model.parameters())
        if not p.is_cuda:
            raise _lib.D3fkError("Sampler needs the model on a B200 (sm_100a) CUDA device")
        self.model, self.device = model, p.device
        self.B, self.H, self.W, self.n_steps = batch, height, width, n_steps
        self.r_start, self.eta, self.seed = float(r_start), float(eta), int(seed)
        self.solver, self.schedule = solver, schedule
        self.multistep = solver == "dpmpp_2m"
        if r_start <= 0:
            self.grid = [0.0] * (n_steps + 1)
        elif schedule == "linear":
            self.grid = noise_ratio_grid(n_steps, r_start)
        else:
            self.grid = noise_ratio_grid(n_steps, r_start, kind=schedule, r_min=r_min)
        was_training = model.training
        model.eval()
        self.x = torch.zeros(batch, 3, height, width, dtype=torch.float32, device=self.device)
        self.x0_hat = torch.zeros_like(self.x)
        self.plan = model._acquire_plan(self.x, training=False)
        self.plan.pending_backward = True        # reserve this plan instance for the sampler
        model.train(was_training)
        table = dpmpp_2m_coef_table(self.grid, eta) if self.multistep else posterior_coef_table(self.grid, eta)
        self.coef_table = torch.tensor(table, dtype=torch.float32, device=self.device).contiguous()
        # 2M: the previous step's x0_hat (the kernel copies x0_hat here; the first step's c = 0 never reads it)
        self.x0_prev = torch.zeros_like(self.x) if self.multistep else None
        self.masked = bool(masked)
        # the source and mask buffers the masked posterior ops point at (run() copies its inputs into them)
        self.src = torch.zeros_like(self.x) if self.masked else None
        self.mask = torch.zeros(batch, 1, height, width, dtype=torch.float32, device=self.device) if self.masked else None
        self.step = torch.zeros(1, dtype=torch.int32, device=self.device)
        if chains is None:
            chains = int(os.environ.get("D3FK_SAMPLER_CHAINS", "1"))
        while chains > 1 and (batch % chains or batch // chains < 1):
            chains -= 1
        self.chains = max(1, chains)
        self.steps_per_graph = steps_per_graph if n_steps % steps_per_graph == 0 else 1
        b = batch // self.chains
        self.chain_plans, self.chain_steps, self.chain_ops = [], [], []
        self.kernels_per_step = 0
        for c in range(self.chains):
            xs, hs = self.x[c * b:(c + 1) * b], self.x0_hat[c * b:(c + 1) * b]
            plan = self.plan if self.chains == 1 else model._new_plan(xs, training=False)
            step = self.step if self.chains == 1 else torch.zeros(1, dtype=torch.int32, device=self.device)
            ops = list(plan.fwd_ops)
            op_params(ops[plan.in_op_index]).src = xs.data_ptr()
            op_params(ops[plan.out_op_index]).out_nchw = hs.data_ptr()
            masked = {}
            if self.masked:
                masked = dict(src=self.src[c * b:(c + 1) * b].data_ptr(), mask=self.mask[c * b:(c + 1) * b].data_ptr(),
                              chw=3 * height * width, hw=height * width)
            # independent Philox streams per chain (the kernel's counter is the element index within its own sub-batch)
            post = dict(n=xs.numel(), x=xs.data_ptr(), x0_hat=hs.data_ptr(), coef_table=self.coef_table.data_ptr(),
                        step=step.data_ptr(), seed=self.seed + 0x9E3779B1 * c, offset=0, **masked)
            if self.multistep:
                ops.append(make_op(_lib.OP_POSTERIOR_2M, base=post, x0_prev=self.x0_prev[c * b:(c + 1) * b].data_ptr()))
            else:
                ops.append(make_op(_lib.OP_POSTERIOR, **post))
            ops.append(make_op(_lib.OP_INC, p0=step.data_ptr(), n=1))
            self.kernels_per_step += len(ops)
            self.chain_plans.append(plan)
            self.chain_steps.append(step)
            self.chain_ops.append(_lib.OpList(ops * self.steps_per_graph))
        self.step_ops = self.chain_ops[0]
        self.side = [torch.cuda.Stream(self.device) for _ in range(self.chains - 1)]
        self.graph = None
        self.use_graph = use_graph
        self._weights_version = None

    def refresh_weights(self):
        """Re-pack bf16 weights and re-fold BN if the model's parameters changed since the last call."""
        ver = self.model._weights_version()
        if ver != self._weights_version:
            stream = torch.cuda.current_stream(self.device).cuda_stream
            for plan in {id(p): p for p in [self.plan] + self.chain_plans}.values():
                plan.run_pack(stream)
            self._weights_version = ver

    def _run_chains(self):
        """One graph's worth of steps of every chain: chain 0 on the current stream, the others forked onto side streams
        and joined back (fork / join are event waits, so this records as parallel graph branches under capture)."""
        cur = torch.cuda.current_stream(self.device)
        for c in range(1, self.chains):
            self.side[c - 1].wait_stream(cur)
        self.chain_ops[0].run(cur.cuda_stream)
        for c in range(1, self.chains):
            self.chain_ops[c].run(self.side[c - 1].cuda_stream)
        for s in self.side:
            cur.wait_stream(s)

    def _capture(self):
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):                  # warm-up launch outside capture
            self._run_chains()
        torch.cuda.current_stream(self.device).wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._run_chains()
        self.graph = g

    @torch.no_grad()
    def run(self, x_start=None, noises=None, src=None, mask=None, known_noises=None):
        """x_start: state at ratio r_start ([B,3,H,W] fp32; default: Philox N(0,1) when r_start == 1).
        noises: optional [n_steps,B,3,H,W] (eta > 0 parity runs; forces the eager path).  Returns x_0.
        Masked sampler: src [B,3,H,W] (the image to keep outside the mask) and mask (see functional.normalize_mask) are
        required; x_start defaults to src noised to r_start (Philox N(0,1) at r_start == 1, as unmasked).  known_noises:
        optional [n_steps,B,3,H,W], the noise of the known region at each step (forces the eager path, as noises does; the
        eager path otherwise draws the graph's in-kernel known noise)."""
        if self.masked != (src is not None and mask is not None) or (not self.masked and known_noises is not None):
            raise ValueError("a masked Sampler needs src and mask (and an unmasked one takes neither, nor known_noises)")
        eager = noises is not None or known_noises is not None
        self.refresh_weights()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        if self.use_graph and self.graph is None and not eager:
            self._capture()                      # (its warm-up launch scribbles on self.x: capture first)
        if self.masked:
            self.src.copy_(src)
            self.mask.copy_(normalize_mask(mask, self.B, self.H, self.W))
        if x_start is None:
            # (q_sample at ratio 1 is the noise alone: the masked start at r_start == 1 is the unmasked one)
            base = self.src if self.masked else torch.zeros_like(self.x)
            r0 = max(self.r_start, 0.0) if self.masked else 1.0
            self.x.copy_(q_sample(base, 1.0, seed=self.seed ^ 0x5EED, fixed_r=r0))
        else:
            self.x.copy_(x_start)
        if eager:
            for i in range(self.n_steps):
                self.plan.run_forward(self.x, self.x0_hat, stream)
                r_prev = self.grid[i + 1] if self.grid[i] > 0 else 0.0
                z = None if noises is None else noises[i]
                if self.multistep:
                    msk = dict(src=self.src, mask=self.mask,
                               known_noise=None if known_noises is None else known_noises[i]) if self.masked else {}
                    dpmpp_2m_step_(self.x, self.x0_hat, self.x0_prev, self.grid[i - 1] if i > 0 else None, self.grid[i],
                                   r_prev, z=z, eta=self.eta, seed=self.seed, offset=i, **msk)
                elif self.masked:
                    posterior_step_(self.x, self.x0_hat, self.grid[i], r_prev, z=z, eta=self.eta, seed=self.seed,
                                    offset=i, src=self.src, mask=self.mask,
                                    known_noise=None if known_noises is None else known_noises[i])
                else:
                    posterior_step_(self.x, self.x0_hat, self.grid[i], r_prev, z=z, eta=self.eta)
            return self.x.clone()
        for st in self.chain_steps:
            st.zero_()
        for _ in range(self.n_steps // self.steps_per_graph):
            if self.use_graph:
                self.graph.replay()
            else:
                self._run_chains()
        return self.x.clone()

    def launches_per_run(self):
        return self.kernels_per_step * self.n_steps


@torch.no_grad()
def sample(model, x_start, n_steps, r_start=1.0, eta=0.0, seed=0, noises=None, use_graph=True, solver="posterior",
           schedule=None):
    B, _, H, W = x_start.shape
    return Sampler(model, B, H, W, n_steps, r_start, eta, seed, use_graph, solver=solver,
                   schedule=schedule).run(x_start, noises)


@torch.no_grad()
def swap_face(model, real, n_steps=1, r_start=0.0, eta=0.0, seed=0, mask=None, solver="posterior", schedule=None):
    """Push `real` (identity A, normalised to [-1,1]) toward the identity `model` was trained on.
    n_steps=1, r_start=0 reproduces the reference exactly: fake = model(real)
    (d3f/train_deep_fake/lit_module.py:189,266).  r_start>0 noises the source to that ratio first and
    runs the iterative sampler from there.
    mask ([H,W], [1,1,H,W] or [B,1,H,W]; 1 = swap, 0 = keep `real`, fractions feather): r_start <= 0 gives the composite
    m*model(real) + (1 - m)*real; r_start > 0 runs the masked sampler, which keeps the source outside the mask at every
    step, so the swapped region is generated in context.  Where m == 0 the result is `real` exactly.
    solver / schedule: as Sampler's ("dpmpp_2m" on its logsnr grid reaches at 10-20 steps what the first-order update
    needs about twice the steps for)."""
    if r_start <= 0.0:
        was = model.training
        model.eval()
        out = model(real)
        model.train(was)
        if mask is None:
            return out
        B, _, H, W = real.shape
        return composite_(out, real, normalize_mask(mask, B, H, W).to(out.device))
    if mask is not None:
        B, _, H, W = real.shape
        return Sampler(model, B, H, W, n_steps, r_start, eta, seed, masked=True, solver=solver,
                       schedule=schedule).run(src=real, mask=mask)
    # the start noise comes from a Philox key of its own (as Sampler.run's does): with the sampler's key the first ancestral
    # z (eta > 0; posterior step 0 draws philox(seed, element, offset 0)) would be the very noise the source was noised with
    x_start = q_sample(real, 1.0, seed=seed ^ 0x5EED, fixed_r=r_start)
    return sample(model, x_start, n_steps, r_start=r_start, eta=eta, seed=seed, solver=solver, schedule=schedule)
