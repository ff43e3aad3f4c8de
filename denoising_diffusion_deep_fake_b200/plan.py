"""Op-list plans for the resnet34 U-Net (smp.Unet restated in SURVEY Appendix A).

A plan is built once per (batch, H, W, dtype, variant) and owns every intermediate buffer; running
it is ONE call into libd3fk (`d3fk_run`) that enqueues the whole forward (or backward) on the
current CUDA stream — no tracing compiler, no per-layer Python in the hot loop, CUDA-graph safe.

Topology follows torchvision/models/resnet.py:89-105,197-205,266-278 (encoder) and smp's
UnetDecoder / DecoderBlock / SegmentationHead (SURVEY Appendix A1); the call being replaced is
`self.model(image_noisy)` at d3f/train_denoiser/lit_module.py:117 and its autograd backward.

Variants: the training plan (batch statistics, backward), the eval plan (BatchNorm folded into the convolutions, forward only)
and the frozen-BN plan (`frozen=True`: BatchNorm on its running statistics as in eval mode, nothing updates them, with a
backward — eval-mode autograd).  `want_dx=True` adds the input gradient to a plan's backward: the stem's dgrad, written as fp32
NCHW into the pointer `run_backward(dx=...)` patches in.
"""
import os

import torch

from . import _lib
from ._lib import make_op, op_params

# D3FK_FUSE_BNBW=<elements>: fold BN-backward's reduction into the epilogue of the dgrad that produces the gradient, for
# layers whose BN tensor has at most that many elements (1 = every layer, 0 = never).  On the big decoder-tail / stem tensors
# the per-lane x / act loads lengthen the dgrad epilogue by more than the removed (HBM-bound) reduction pass costs; on the
# deep, latency-bound layers the removed kernel boundary wins.
_f = int(os.environ.get("D3FK_FUSE_BNBW", "1100000"))    # measured on B200: 4.425 ms/step vs 4.475 unfused, 4.58 all fused
FUSE_BN_BWD_MAX_ELEMS = (1 << 62) if _f == 1 else _f
# D3FK_WGRAD_GROUP=1: one weight-gradient launch per group of identically shaped encoder layers (D3FK_OP_WGRAD_GROUP) instead
# of one per convolution.  Measured: -0.33 ms of GPU work per step, but no change of the step time (the weight gradients are
# hidden behind the latency-bound main chain either way, and the last group lengthens the tail) - opt-in.
GROUP_WGRAD = os.environ.get("D3FK_WGRAD_GROUP", "0") == "1"
# D3FK_WGRAD_GROUP_SIZE=n (with D3FK_WGRAD_GROUP=1): flush a group as soon as it holds n problems instead of at the end of the
# stage (0: whole stage) - the grouped launch then starts earlier, behind the n-th BatchNorm backward.
GROUP_WGRAD_SIZE = int(os.environ.get("D3FK_WGRAD_GROUP_SIZE", "0"))

# Materialise upsample + concat for EVERY decoder block whose channel count is a multiple of 64 (blocks 0-2: 768 / 384 / 192
# channels), so that conv1 and its weight gradient are TMA-fed instead of gathering through the upsample: three small streaming
# passes (17 us) buy 49 -> 30, 40 -> 26 and 41 -> 26 us on the forward convolutions (eval: 43 -> 22, 34 -> 15, 29 -> 19) and TMA weight
# gradients: 3.63 -> 3.59 ms per training step, 0.817 -> 0.767 ms per sampling step.  D3FK_UPCAT_ALL=0: gather through the upsample.
UPCAT_ALL = os.environ.get("D3FK_UPCAT_ALL", "1") == "1"

# The downsample branch of a stage's first block on a branch stream of d3fk_run (0: everything on the main chain).
BRANCH_LANE = int(os.environ.get("D3FK_BRANCH_LANE", "1"))

BN_EPS = 1e-5
BN_MOMENTUM = 0.1
SPLITK_WS_BYTES = 64 << 20
CIN_PAD = 8  # the RGB input is zero padded to 8 channels (16-byte bf16 gather chunks)
DY_PAD = 16  # the 3-channel head gradient is zero padded to 16 channels (one UMMA K step: the slab dgrad path)


class ConvSpec:
    def __init__(self, name, cin, cout, k, stride, pad, bn=None, bias=False):
        self.name, self.cin, self.cout, self.k, self.stride, self.pad = name, cin, cout, k, stride, pad
        self.bn = bn          # state_dict prefix of the BatchNorm2d that follows (None for the head)
        self.bias = bias


def unet_layers():
    """Static description of the 47 convolutions in forward order, grouped by stage."""
    stem = ConvSpec("encoder.conv1", 3, 64, 7, 2, 3, bn="encoder.bn1")
    stages = []
    cin = 64
    for li, (cout, nblocks) in enumerate(((64, 3), (128, 4), (256, 6), (512, 3)), start=1):
        blocks = []
        for bi in range(nblocks):
            stride = 2 if (bi == 0 and li > 1) else 1
            p = f"encoder.layer{li}.{bi}"
            blk = {
                "conv1": ConvSpec(f"{p}.conv1", cin, cout, 3, stride, 1, bn=f"{p}.bn1"),
                "conv2": ConvSpec(f"{p}.conv2", cout, cout, 3, 1, 1, bn=f"{p}.bn2"),
                "down": ConvSpec(f"{p}.downsample.0", cin, cout, 1, stride, 0, bn=f"{p}.downsample.1")
                if (stride != 1 or cin != cout) else None,
            }
            blocks.append(blk)
            cin = cout
        stages.append(blocks)
    dec = []
    for i, (ci, cs, co) in enumerate(((512, 256, 256), (256, 128, 128), (128, 64, 64), (64, 64, 32), (32, 0, 16))):
        p = f"decoder.blocks.{i}"
        dec.append({
            "cin": ci, "cskip": cs, "cout": co,
            "conv1": ConvSpec(f"{p}.conv1.0", ci + cs, co, 3, 1, 1, bn=f"{p}.conv1.1"),
            "conv2": ConvSpec(f"{p}.conv2.0", co, co, 3, 1, 1, bn=f"{p}.conv2.1"),
        })
    head = ConvSpec("segmentation_head.0", 16, 3, 3, 1, 1, bias=True)
    return stem, stages, dec, head


def all_convs():
    stem, stages, dec, head = unet_layers()
    out = [stem]
    for blocks in stages:
        for b in blocks:
            out.append(b["conv1"])
            out.append(b["conv2"])
            if b["down"] is not None:
                out.append(b["down"])
    for d in dec:
        out += [d["conv1"], d["conv2"]]
    out.append(head)
    return out


def backward_param_order():
    """Parameter names in the order their gradients become final during backward
    (head, decoder 4..0, layer4..layer1 reversed, stem) — the flat gradient arena and the
    data-parallel allreduce buckets follow this order."""
    stem, stages, dec, head = unet_layers()
    names = [head.name + ".weight", head.name + ".bias"]

    def conv_bn(c):
        return [c.name + ".weight", c.bn + ".weight", c.bn + ".bias"]

    for d in reversed(dec):
        names += conv_bn(d["conv2"]) + conv_bn(d["conv1"])
    for blocks in reversed(stages):
        for b in reversed(blocks):
            names += conv_bn(b["conv2"])
            if b["down"] is not None:
                names += conv_bn(b["down"])
            names += conv_bn(b["conv1"])
    names += conv_bn(stem)
    return names


class T:
    """An NHWC activation buffer owned by the plan."""

    def __init__(self, plan, B, H, W, C, dtype=None):
        self.B, self.H, self.W, self.C = B, H, W, C
        self.t = torch.empty((B, H, W, C), dtype=dtype or plan.tdtype, device=plan.device)
        self.ptr = self.t.data_ptr()
        self.ld = C
        self.count = B * H * W


class UnetPlan:
    def __init__(self, params, buffers, B, H, W, dtype, device, training, grad_arena=None, grad_offsets=None, frozen=False,
                 want_dx=False):
        """params/buffers: dict name -> tensor (the module's own parameters / BN buffers, fp32).  frozen (with training=False):
        the frozen-BN plan.  want_dx (plans with a backward): the backward also produces the gradient of the input image."""
        if H % 32 or W % 32:
            raise RuntimeError(f"Wrong input shape height={H}, width={W}. Expected image height and width "
                               f"divisible by 32.")
        self.B, self.H, self.W = B, H, W
        self.dtype = dtype
        self.tdtype = torch.float32 if dtype == _lib.F32 else torch.bfloat16
        self.device = torch.device(device)
        self.training = training
        self.frozen = bool(frozen) and not training
        self.has_backward = training or self.frozen
        if want_dx and not self.has_backward:
            raise ValueError("want_dx needs a plan with a backward (training or frozen)")
        self.want_dx = bool(want_dx)
        self.params, self.buffers = params, buffers
        self.keep = []          # every tensor the op lists point into
        self.generation = 0
        self.pending_backward = False
        self.stem, self.stages, self.dec, self.head = unet_layers()
        self.convs = all_convs()
        self.param_ptrs = {}
        self._alloc_weights()
        self._alloc_bn()
        # fp32 scratch for split-K convolutions (deep layers whose output tiles cannot fill 148 SMs)
        self.ws = self._new((SPLITK_WS_BYTES // 4,), torch.float32) if dtype == _lib.BF16 else None
        self.grad_arena, self.grad_offsets = (grad_arena, grad_offsets) if self.has_backward else (None, None)
        self.pack_ops = _lib.OpList(self._build_pack())
        self.prepacked_version = None   # Unet._weights_version() the packed operands were last produced for (train.StepOverlap)
        self.saved = {}
        fwd = self._build_forward()
        self.fwd_ops = _lib.OpList(fwd)
        self.bwd_segments = None
        if self.has_backward:
            self.bwd_segments = [_lib.OpList(seg) for seg in self._build_backward()]
        self._record_param_ptrs()

    # ------------------------------------------------------------------ allocation helpers
    def _new(self, shape, dtype):
        t = torch.zeros(shape, dtype=dtype, device=self.device)
        self.keep.append(t)
        return t

    def _alloc_weights(self):
        self.w_fwd, self.w_dgrad = {}, {}
        for c in self.convs:
            cin_pad = CIN_PAD if c.cin == 3 else c.cin
            cout_pad = DY_PAD if c.cout == 3 else c.cout
            taps = c.k * c.k
            self.w_fwd[c.name] = self._new((c.cout, taps * cin_pad), self.tdtype)
            if self.has_backward and (c.name != self.stem.name or self.want_dx):
                # the stem's dgrad operand [3][7][7][64] only where the input gradient is wanted (compared by name: all_convs()
                # builds its own ConvSpec objects)
                self.w_dgrad[c.name] = self._new((c.cin, taps * cout_pad), self.tdtype)
        # bf16 engine: the 7x7 / stride-2 stem runs as a space-to-depth convolution (conv mode 2, include/d3fk.h) whenever
        # its 128-pixel output tile is a (w, h, n) box — K = 256 by TMA instead of K = 392 by per-thread gather (65 -> 25 us)
        self.stem_s2d = self.dtype == _lib.BF16 and self._stem_box_ok(self.H // 2, self.W // 2)
        self.w_stem_s2d = self._new((self.stem.cout, 256), self.tdtype) if self.stem_s2d else None

    @staticmethod
    def _stem_box_ok(Ho, Wo):
        """tma_box() of csrc/conv_tc.cu for the stem's output: 128 consecutive pixels form an axis-aligned (w, h, n) box."""
        bw = min(Wo, 128)
        if 128 % bw or Wo % bw:
            return False
        bh = min(128 // bw, Ho)
        if (128 // bw) % bh or Ho % bh:
            return False
        bn = 128 // (bw * bh)
        return not (bw < Wo and bh != 1) and not (bh < Ho and bn != 1) and bn <= 256

    def _alloc_bn(self):
        bns = [c for c in self.convs if c.bn]
        total = sum(c.cout for c in bns)
        self.bn_f32 = self._new((8, total), torch.float32)      # scale, shift, mean, invstd, coef[3], spare
        # [fwd|bwd][per-BN (sum, sumsq) ... | one 8-byte slot per BN: grid-barrier counter of the fused conv+BN kernel]
        self.stats = self._new((2, 2 * total + len(bns)), torch.float64)
        self.bn_off, self.bn_barrier = {}, {}
        off = 0
        for i, c in enumerate(bns):
            self.bn_off[c.bn] = off
            self.bn_barrier[c.bn] = self.stats[0].data_ptr() + 8 * (2 * total + i)
            off += c.cout

    def _bnptr(self, bn, row, C):
        return self.bn_f32[row].data_ptr() + 4 * self.bn_off[bn]

    def _bn_common(self, c):
        bn, C = c.bn, c.cout
        off = self.bn_off[bn]
        coef = self._new((3, C), torch.float32)
        return dict(
            dtype=self.dtype, C=C, eps=BN_EPS, momentum=BN_MOMENTUM,
            gamma=self.params[bn + ".weight"].data_ptr(), beta=self.params[bn + ".bias"].data_ptr(),
            running_mean=self.buffers[bn + ".running_mean"].data_ptr(),
            running_var=self.buffers[bn + ".running_var"].data_ptr(),
            num_batches_tracked=self.buffers[bn + ".num_batches_tracked"].data_ptr(),
            scale=self._bnptr(bn, 0, C), shift=self._bnptr(bn, 1, C), mean=self._bnptr(bn, 2, C),
            invstd=self._bnptr(bn, 3, C), coef=coef.data_ptr(),
            stats=self.stats[0].data_ptr() + 8 * 2 * off, bstats=self.stats[1].data_ptr() + 8 * 2 * off,
        )

    def _record_param_ptrs(self):
        self.param_ptrs = {n: p.data_ptr() for n, p in self.params.items()}
        self.param_ptrs.update({n: b.data_ptr() for n, b in self.buffers.items()})

    def params_moved(self):
        for n, p in self.params.items():
            if self.param_ptrs.get(n) != p.data_ptr():
                return True
        for n, b in self.buffers.items():
            if self.param_ptrs.get(n) != b.data_ptr():
                return True
        return False

    # ------------------------------------------------------------------ weight packing / BN folding
    def _build_pack(self):
        """Pack ops, grouped by gradient bucket (= backward segment): `pack_bucket_ops[i]` re-packs exactly the layers whose
        master weights bucket i of the flat arena holds, so a trainer can re-pack a bucket as soon as its Adam update has
        run, while the rest of backward is still executing (train.StepOverlap)."""
        import bisect
        import ctypes
        ops = []
        if self.grad_offsets is not None:
            stage_first = ["segmentation_head.0.weight", "encoder.layer4.2.conv2.weight", "encoder.layer3.5.conv2.weight",
                           "encoder.layer2.3.conv2.weight", "encoder.layer1.2.conv2.weight"]
            starts = [self.grad_offsets[n] for n in stage_first]
            bucket_of = lambda c: bisect.bisect_right(starts, self.grad_offsets[c.name + ".weight"]) - 1
            n_buckets = len(starts)
        else:
            bucket_of = lambda c: 0
            n_buckets = 1
        groups = [[] for _ in range(n_buckets)]
        for c in self.convs:
            groups[bucket_of(c)].append(c)
        packs, spans = [], []
        for group in groups:
            blocks, first = 0, len(packs)
            for c in group:
                cin_pad = CIN_PAD if c.cin == 3 else c.cin
                cout_pad = DY_PAD if c.cout == 3 else c.cout
                wd = self.w_dgrad.get(c.name)
                assert c.k * c.k * min(c.cin, 32) <= 288, "pack_all tile: taps * min(Cin, 32) must be <= 288"
                packs.append(make_op(_lib.OP_PACK, dtype=self.dtype, Cout=c.cout, Cin=c.cin, kh=c.k, kw=c.k,
                                     cin_pad=cin_pad, cout_pad=cout_pad, blk0=blocks,
                                     w=self.params[c.name + ".weight"].data_ptr(),
                                     w_fwd=self.w_fwd[c.name].data_ptr(),
                                     w_dgrad=wd.data_ptr() if wd is not None else None))
                blocks += -(-c.cout // 32) * -(-c.cin // 32)
            spans.append((first, len(packs) - first, blocks))
        # one launch per bucket: the descriptors live in a device table (blk0 restarts at each bucket)
        table = (_lib.PackParams * len(packs))(*[op_params(o) for o in packs])
        raw = torch.frombuffer(bytearray(bytes(table)), dtype=torch.uint8).clone()
        self.pack_table = raw.to(self.device)
        self.keep.append(self.pack_table)
        self.pack_bucket_ops = []
        for first, count, blocks in spans:
            if count == 0:
                self.pack_bucket_ops.append(None)
                continue
            op = make_op(_lib.OP_PACK_ALL, p0=self.pack_table.data_ptr() + first * ctypes.sizeof(_lib.PackParams),
                         n=(blocks << 17) | (count << 1) | (1 if self.dtype == _lib.BF16 else 0))
            ops.append(op)
            bucket_ops = [op]
            if self.stem_s2d and len(self.pack_bucket_ops) == bucket_of(self.stem):
                stem_op = make_op(_lib.OP_PACK_STEM, dtype=self.dtype, Cout=self.stem.cout, Cin=3, kh=7, kw=7, cin_pad=4,
                                  cout_pad=self.stem.cout, w=self.params[self.stem.name + ".weight"].data_ptr(),
                                  w_fwd=self.w_stem_s2d.data_ptr())
                ops.append(stem_op)
                bucket_ops.append(stem_op)
            self.pack_bucket_ops.append(_lib.OpList(bucket_ops))
        if not self.training:
            # frozen plans also publish the running statistics as mean / invstd: the backward's xhat rows
            keys = ("dtype", "C", "eps", "gamma", "beta", "running_mean", "running_var", "scale", "shift") + \
                (("mean", "invstd") if self.frozen else ())
            for c in self.convs:
                if c.bn:
                    ops.append(make_op(_lib.OP_BN_FOLD, **{k: v for k, v in self._bn_common(c).items() if k in keys}))
        return ops

    # ------------------------------------------------------------------ forward
    def _conv_fields(self, c, src0, src1=None, up0=0, out=None, relu=0, res=None, stats=False, out_nchw=None,
                     affine=False, override=None):
        Hi = src0.H * (2 if up0 else 1)
        Wi = src0.W * (2 if up0 else 1)
        Ho = (Hi + 2 * c.pad - c.k) // c.stride + 1
        Wo = (Wi + 2 * c.pad - c.k) // c.stride + 1
        f = dict(dtype=self.dtype, mode=0, src0=src0.ptr, c0=src0.C, ld0=src0.ld, up0=up0,
                 B=self.B, Hi=Hi, Wi=Wi, Ho=Ho, Wo=Wo, kh=c.k, kw=c.k, stride=c.stride, pad=c.pad,
                 w=self.w_fwd[c.name].data_ptr(), Cout=c.cout, relu=relu)
        if self.ws is not None:
            f.update(ws=self.ws.data_ptr(), ws_bytes=SPLITK_WS_BYTES)
        if src1 is not None:
            f.update(src1=src1.ptr, c1=src1.C, ld1=src1.ld)
        if out is not None:
            f.update(out=out.ptr, ldo=out.ld)
        if out_nchw is not None:
            f.update(out_nchw=out_nchw)
        if res is not None:
            f.update(res=res.ptr, ldr=res.ld)
        if stats:
            f.update(stats=self.stats[0].data_ptr() + 8 * 2 * self.bn_off[c.bn])
        if affine:
            f.update(scale=self._bnptr(c.bn, 0, c.cout), shift=self._bnptr(c.bn, 1, c.cout))
        if override:
            f.update(override)
        return f

    def _conv_op(self, c, src0, src1=None, up0=0, out=None, relu=0, res=None, stats=False, out_nchw=None,
                 affine=False, lane=0, override=None):
        f = self._conv_fields(c, src0, src1, up0, out, relu, res, stats, out_nchw, affine, override)
        return make_op(_lib.OP_CONV, lane=lane, **f), f["Ho"], f["Wo"]

    def _conv_bn_act(self, ops, c, src0, src1=None, up0=0, relu=1, res=None, lane=0, override=None):
        """conv -> BN -> (+res) -> ReLU.  Train: raw conv output + batch statistics in the conv epilogue,
        finalize, one fused apply pass.  Eval: BN folded into the conv epilogue.  Frozen: the raw conv output is kept for
        backward and one apply pass uses the folded scale / shift (no statistics, no barrier).  Returns the activation.
        lane != 0: the op runs on a branch stream of d3fk_run (always in its two-kernel form: a branch never waits on a
        grid-wide barrier)."""
        Hi = src0.H * (2 if up0 else 1)
        Ho = (Hi + 2 * c.pad - c.k) // c.stride + 1
        Wi = src0.W * (2 if up0 else 1)
        Wo = (Wi + 2 * c.pad - c.k) // c.stride + 1
        act = T(self, self.B, Ho, Wo, c.cout)
        self.keep.append(act.t)
        if not self.has_backward:
            op, _, _ = self._conv_op(c, src0, src1, up0, out=act, relu=relu, res=res, affine=True, lane=lane, override=override)
            ops.append(op)
            return act
        raw = T(self, self.B, Ho, Wo, c.cout)
        self.keep.append(raw.t)
        conv_fields = self._conv_fields(c, src0, src1, up0, out=raw, stats=not self.frozen, override=override)
        bn = self._bn_common(c)
        bn.update(count=raw.count, relu=relu, x=raw.ptr, ldx=raw.ld, y=act.ptr, ldy=act.ld)
        if self.frozen:
            bn.update(stats=None, frozen=1)
        if res is not None:
            bn.update(res=res.ptr, ldr=res.ld)
        fwd_fields = {k: v for k, v in bn.items() if k not in ("bstats", "coef", "frozen")}
        # ONE op: conv + BN finalize + normalise (+residual) + ReLU — fused into the conv kernel where the layer qualifies
        ops.append(make_op(_lib.OP_CONV_BN, lane=lane, conv=conv_fields, bn=fwd_fields,
                           barrier=None if (lane or self.frozen) else self.bn_barrier[c.bn]))
        self.saved[c.name] = dict(src0=src0, src1=src1, up0=up0, raw=raw, act=act, relu=relu, bn=bn, res=res)
        return act

    def _build_forward(self):
        ops = []
        B, H, W = self.B, self.H, self.W
        if self.training:
            ops.append(make_op(_lib.OP_MEMSET, p0=self.stats[0].data_ptr(), n=self.stats[0].numel() * 8))
        self.x8 = T(self, B, H, W, CIN_PAD)
        self.keep.append(self.x8.t)
        self.in_op_indices = []           # every op that reads the caller's NCHW input (run_forward patches their .src)
        stem_override = None
        if self.stem_s2d:
            # padded space-to-depth image [B][H/2][W/2 + 3][16] (zero-initialised: the pad pixels / 4th channel are never written)
            self.xs2d = self._new((B, H // 2, W // 2 + 3, 16), self.tdtype)
            self.in_op_indices.append(len(ops))
            ops.append(make_op(_lib.OP_NCHW2S2D, dtype=self.dtype, B=B, C=3, H=H, W=W, cpad=4, src=None, dst=self.xs2d.data_ptr()))
            stem_override = dict(mode=2, src0=self.xs2d.data_ptr(), c0=64, c1=0, ld0=16, up0=0, Hi=H // 2, Wi=W // 2, kh=4, kw=1,
                                 stride=1, pad=2, w=self.w_stem_s2d.data_ptr())
        if not self.stem_s2d:                       # the 8-channel NHWC image of the gather-form stem (and its weight gradient)
            self.in_op_indices.append(len(ops))
            ops.append(make_op(_lib.OP_NCHW2NHWC, dtype=self.dtype, B=B, C=3, H=H, W=W, cpad=CIN_PAD, src=None,
                               dst=self.x8.ptr))
        self.in_op_index = self.in_op_indices[0]
        f1 = self._conv_bn_act(ops, self.stem, self.x8, override=stem_override)
        p1 = T(self, B, f1.H // 2, f1.W // 2, 64)
        self.keep.append(p1.t)
        self.pool_idx = self._new((B, p1.H, p1.W, 64), torch.uint8) if self.has_backward else None
        ops.append(make_op(_lib.OP_MAXPOOL_FWD, dtype=self.dtype, B=B, H=f1.H, W=f1.W, C=64, x=f1.ptr, ldx=f1.ld,
                           y=p1.ptr, ldy=p1.ld, idx=self.pool_idx.data_ptr() if self.has_backward else None))
        self.f1, self.p1 = f1, p1
        x = p1
        feats = [f1]
        self.block_io = []
        for blocks in self.stages:
            for b in blocks:
                idn = x
                if b["down"] is not None:
                    # the 1x1 / stride-2 downsample branch is independent of conv1 -> BN -> ReLU until the residual add
                    # (torchvision BasicBlock.forward, resnet.py:89-105): it runs on branch lane 1, next to conv1
                    idn = self._conv_bn_act(ops, b["down"], x, relu=0, lane=BRANCH_LANE)
                a1 = self._conv_bn_act(ops, b["conv1"], x)
                if b["down"] is not None and BRANCH_LANE:
                    ops.append(make_op(_lib.OP_JOIN, n=BRANCH_LANE))
                out = self._conv_bn_act(ops, b["conv2"], a1, relu=1, res=idn)
                self.block_io.append((b, x, a1, idn, out))
                x = out
            feats.append(x)
        # feats = [f1, f2, f3, f4, f5]
        self.feats = feats
        skips = [feats[3], feats[2], feats[1], feats[0], None]
        x = feats[4]
        self.dec_io = []
        for d, skip in zip(self.dec, skips):
            ctot = x.C + (skip.C if skip is not None else 0)
            if (2 * x.W >= 16 and ctot in (16, 32, 64, 128)) or (UPCAT_ALL and ctot % 64 == 0):
                # materialise upsample + concat once (one streaming pass) so conv1 — and its weight gradient — run on the
                # slab path (each activation row read 3x by TMA) or the TMA-fed generic path instead of a 9x per-thread gather
                # through the upsample
                cat = T(self, B, 2 * x.H, 2 * x.W, ctot)
                self.keep.append(cat.t)
                f = dict(dtype=self.dtype, B=B, H=cat.H, W=cat.W, c0=x.C, ld0=x.ld, ldo=cat.ld, src0=x.ptr, out=cat.ptr)
                if skip is not None:
                    f.update(c1=skip.C, ld1=skip.ld, src1=skip.ptr)
                ops.append(make_op(_lib.OP_UPCAT, **f))
                a1 = self._conv_bn_act(ops, d["conv1"], cat)
                self.dec_io.append((d, x, skip, a1, None, cat))
            else:
                a1 = self._conv_bn_act(ops, d["conv1"], x, src1=skip, up0=1)
                self.dec_io.append((d, x, skip, a1, None, None))
            out = self._conv_bn_act(ops, d["conv2"], a1)
            self.dec_io[-1] = self.dec_io[-1][:4] + (out, self.dec_io[-1][5])
            x = out
        self.dec_out = x
        self.out_op_index = len(ops)
        op, _, _ = self._conv_op(self.head, x, out_nchw=0)
        op_params(op).shift = self.params[self.head.name + ".bias"].data_ptr()
        ops.append(op)
        return ops

    # ------------------------------------------------------------------ backward
    def _gptr(self, name):
        return self.grad_arena.data_ptr() + 4 * self.grad_offsets[name]

    def _wgrad_op(self, c, src0, src1, up0, dy, cout_buf=None, lane=0):
        Hi = src0.H * (2 if up0 else 1)
        Wi = src0.W * (2 if up0 else 1)
        f = dict(dtype=self.dtype, src0=src0.ptr, c0=src0.C, ld0=src0.ld, up0=up0, B=self.B, Hi=Hi, Wi=Wi,
                 Ho=dy.H, Wo=dy.W, kh=c.k, kw=c.k, stride=c.stride, pad=c.pad, dy=dy.ptr, ldy=dy.ld,
                 Cout=dy.C, cin_real=c.cin, cout_real=c.cout, dw=self._gptr(c.name + ".weight"))
        if src1 is not None:
            f.update(src1=src1.ptr, c1=src1.C, ld1=src1.ld)
        return make_op(_lib.OP_WGRAD, lane=lane, **f)

    def _wgrad_ops(self, c, src0, src1, up0, dy, lane=0):
        """Weight-gradient op(s) of one convolution.  A 3x3 / stride-1 layer with 128 input channels and a narrow output
        (decoder block 3 conv1: 128 -> 32 on 262 144 pixels, the largest single kernel of the step through the generic
        kernel's 64-wide tiles) is split into two 64-channel halves of the input — pixel stride unchanged, channel
        offset 64, dW offset 64 * 9 — each of which the slab weight-gradient kernel takes (activations by TMA, read
        3.75x from L2 instead of 9x, no per-thread gather)."""
        if (self.dtype == _lib.BF16 and src1 is None and not up0 and c.k == 3 and c.stride == 1 and c.cin == 128
                and c.cout in (16, 32) and src0.W in (16, 32, 64) and src0.count >= 128 * 148 * 4):
            esz = 2
            ops = []
            for half in range(2):
                f = dict(dtype=self.dtype, src0=src0.ptr + half * 64 * esz, c0=64, ld0=src0.ld, up0=0, B=self.B, Hi=src0.H,
                         Wi=src0.W, Ho=dy.H, Wo=dy.W, kh=3, kw=3, stride=1, pad=1, dy=dy.ptr, ldy=dy.ld, Cout=dy.C,
                         cin_real=c.cin, cout_real=c.cout, dw=self._gptr(c.name + ".weight") + half * 64 * 9 * 4)
                ops.append(make_op(_lib.OP_WGRAD, lane=lane, **f))
            return ops
        return [self._wgrad_op(c, src0, src1, up0, dy, lane=lane)]

    def _wgrad_encoder(self, ops, pending, c, src, dy):
        """Weight gradient of an encoder convolution.  The 3x3 / stride-1 / Cin == Cout convolutions of a ResNet stage are
        identically shaped: they are collected and emitted as ONE grouped launch at the end of the stage's segment
        (D3FK_OP_WGRAD_GROUP) — every dY of the stage is alive until then, the plan never recycles gradient buffers."""
        if GROUP_WGRAD and c.k == 3 and c.stride == 1 and c.cin == c.cout and len(pending) < _lib.WGRAD_GROUP_MAX:
            pending.append((c, src, dy))
            if GROUP_WGRAD_SIZE and len(pending) >= GROUP_WGRAD_SIZE:
                self._flush_wgrad_group(ops, pending)
        else:
            ops.append(self._wgrad_op(c, src, None, 0, dy))

    def _flush_wgrad_group(self, ops, pending):
        if not pending:
            return
        if len(pending) == 1:
            c, src, dy = pending[0]
            ops.append(self._wgrad_op(c, src, None, 0, dy))
        else:
            c, src, dy = pending[0]
            for c2, s2, d2 in pending[1:]:
                assert (c2.k, c2.stride, c2.pad, c2.cin, c2.cout, s2.H, s2.W, s2.C, s2.ld, d2.H, d2.W, d2.C, d2.ld) == \
                       (c.k, c.stride, c.pad, c.cin, c.cout, src.H, src.W, src.C, src.ld, dy.H, dy.W, dy.C, dy.ld)
            base = dict(dtype=self.dtype, c0=src.C, ld0=src.ld, up0=0, B=self.B, Hi=src.H, Wi=src.W, Ho=dy.H, Wo=dy.W,
                        kh=c.k, kw=c.k, stride=c.stride, pad=c.pad, ldy=dy.ld, Cout=dy.C, cin_real=c.cin, cout_real=c.cout)
            ops.append(make_op(_lib.OP_WGRAD_GROUP, base=base, count=len(pending),
                               src0=[s2.ptr for _, s2, _ in pending], dy=[d2.ptr for _, _, d2 in pending],
                               dw=[self._gptr(c2.name + ".weight") for c2, _, _ in pending]))
        pending.clear()

    def _dgrad_op(self, c, dy, out, res=None, row0=0, rows=None, lane=0):
        """dX (= out, channels [row0, row0+rows) of the conv input) from dY through conv c."""
        cout_pad = dy.C
        rows = out.C if rows is None else rows
        wbytes = 4 if self.dtype == _lib.F32 else 2
        f = dict(dtype=self.dtype, mode=1, src0=dy.ptr, c0=dy.C, ld0=dy.ld, B=self.B, Hi=dy.H, Wi=dy.W,
                 Ho=out.H, Wo=out.W, kh=c.k, kw=c.k, stride=c.stride, pad=c.pad,
                 w=self.w_dgrad[c.name].data_ptr() + row0 * c.k * c.k * cout_pad * wbytes, Cout=rows,
                 out=out.ptr, ldo=out.ld)
        if self.ws is not None:
            f.update(ws=self.ws.data_ptr(), ws_bytes=SPLITK_WS_BYTES)
        if res is not None:
            f.update(res=res.ptr, ldr=res.ld)
        return make_op(_lib.OP_CONV, lane=lane, **f)

    def _bn_bwd(self, ops, c, g_act, want_dres=False, lane=0):
        """Backward through BN(+ReLU) of conv c given grad wrt its activation.  Returns (d_raw, g_masked)."""
        sv = self.saved[c.name]
        raw, act = sv["raw"], sv["act"]
        d_raw = T(self, raw.B, raw.H, raw.W, raw.C)
        self.keep.append(d_raw.t)
        bn = dict(sv["bn"])
        bn.update(dy=g_act.ptr, lddy=g_act.ld, act=act.ptr, ldact=act.ld, dx=d_raw.ptr, lddx=d_raw.ld,
                  dgamma=self._gptr(c.bn + ".weight"), dbeta=self._gptr(c.bn + ".bias"))
        g_masked = None
        if want_dres:
            g_masked = T(self, raw.B, raw.H, raw.W, raw.C)
            self.keep.append(g_masked.t)
            bn.update(dres=g_masked.ptr, lddres=g_masked.ld)
        # no residual in the forward: act = relu(raw * scale + shift) exactly, so backward re-derives the ReLU mask from
        # raw (which it streams anyway) and the scale / shift the forward published instead of reading act
        bn["mask_from_x"] = 1 if (sv["res"] is None and sv["relu"]) else 0
        bn.pop("res", None)
        bn.pop("ldr", None)
        fuse = self.dtype == _lib.BF16 and raw.B * raw.H * raw.W * raw.C <= FUSE_BN_BWD_MAX_ELEMS
        prod = self._grad_producer.get(id(g_act)) if fuse else None
        if prod is not None:
            # The gradient arriving here was written (last) by a dgrad convolution: that kernel's epilogue also produces
            # sum(g') and sum(g' * xhat) (d3fk_conv_params.bw_*), so only the apply pass is left of BN backward.
            pp = op_params(prod)
            pp.stats = bn["bstats"]
            pp.bw_x, pp.bw_ldx = raw.ptr, raw.ld
            pp.bw_act, pp.bw_ldact = act.ptr, act.ld
            pp.bw_mean, pp.bw_invstd = bn["mean"], bn["invstd"]
            pp.bw_relu = bn["relu"]
            ops.append(make_op(_lib.OP_BN_BWD_APPLY, lane=lane, **bn))
        else:
            # reduce + apply as ONE op; the apply phase derives its coefficients and writes dgamma / dbeta.  The barrier
            # counter (one-kernel form, opt-in) is cleared by the backward's statistics memset.  Branch lanes: two kernels.
            # Frozen: one streaming pass (dx does not depend on the reductions) and the finalize, no barrier.
            bn["barrier"] = None if (lane or self.frozen) else self.bn_barrier[c.bn] + self.stats.stride(0) * 8
            ops.append(make_op(_lib.OP_BN_BWD, lane=lane, **bn))
        return d_raw, g_masked

    def _newT(self, like, C=None, H=None, W=None):
        t = T(self, like.B, H or like.H, W or like.W, C or like.C)
        self.keep.append(t.t)
        return t

    def _build_backward(self):
        """Returns a list of op-list segments; segment i completes the gradients of bucket i of the flat
        gradient arena (see backward_param_order / Unet.grad_buckets)."""
        B = self.B
        segs = []
        ops = []
        self._grad_producer = {}   # id(gradient buffer) -> the dgrad conv op that wrote it last (None: written by another kind of op)
        ops.append(make_op(_lib.OP_MEMSET, p0=self.grad_arena.data_ptr(), n=self.grad_arena.numel() * 4))
        ops.append(make_op(_lib.OP_MEMSET, p0=self.stats[1].data_ptr(), n=self.stats[1].numel() * 8))
        # ---- head
        self.dy8 = T(self, B, self.H, self.W, DY_PAD)
        self.keep.append(self.dy8.t)
        self.dy_op_index = len(ops)
        # ... and the head's bias gradient (per-channel sums of dY) in the same pass
        ops.append(make_op(_lib.OP_NCHW2NHWC, dtype=self.dtype, B=B, C=3, H=self.H, W=self.W, cpad=DY_PAD, src=None,
                           dst=self.dy8.ptr, chansum=self._gptr(self.head.name + ".bias")))
        ops.append(self._wgrad_op(self.head, self.dec_out, None, 0, self.dy8))
        g = self._newT(self.dec_out)
        ops.append(self._dgrad_op(self.head, self.dy8, g))
        self._grad_producer[id(g)] = ops[-1]
        grad = {id(self.dec_out): g}   # activation buffer -> its (so far accumulated) gradient buffer

        def add_grad(ops, conv, dy, target, row0=0, rows=None, tmp=None, lane=0):
            """dgrad of `conv` into the gradient of `target` (accumulating if one exists)."""
            if tmp is not None:
                ops.append(self._dgrad_op(conv, dy, tmp, row0=row0, rows=rows, lane=lane))
                return
            if id(target) in grad:
                gbuf = grad[id(target)]
                ops.append(self._dgrad_op(conv, dy, gbuf, res=gbuf, row0=row0, rows=rows, lane=lane))
            else:
                gbuf = self._newT(target)
                grad[id(target)] = gbuf
                ops.append(self._dgrad_op(conv, dy, gbuf, row0=row0, rows=rows, lane=lane))
            self._grad_producer[id(gbuf)] = ops[-1]

        # ---- decoder, last block first
        for d, x, skip, a1, out, cat in reversed(self.dec_io):
            d_r2, _ = self._bn_bwd(ops, d["conv2"], grad[id(out)])
            ops.append(self._wgrad_op(d["conv2"], a1, None, 0, d_r2))
            add_grad(ops, d["conv2"], d_r2, a1)
            d_r1, _ = self._bn_bwd(ops, d["conv1"], grad[id(a1)])
            if cat is not None:
                ops += self._wgrad_ops(d["conv1"], cat, None, 0, d_r1)         # the materialised upsample + concat
            else:
                ops.append(self._wgrad_op(d["conv1"], x, skip, 1, d_r1))
            up_tmp = T(self, B, 2 * x.H, 2 * x.W, x.C)
            self.keep.append(up_tmp.t)
            add_grad(ops, d["conv1"], d_r1, None, row0=0, rows=x.C, tmp=up_tmp)
            gx = self._newT(x)
            grad[id(x)] = gx
            ops.append(make_op(_lib.OP_SUMPOOL2, dtype=self.dtype, B=B, H=x.H, W=x.W, C=x.C, dy=up_tmp.ptr,
                               lddy=up_tmp.ld, dx=gx.ptr, lddx=gx.ld))
            self._grad_producer[id(gx)] = None
            if skip is not None:
                add_grad(ops, d["conv1"], d_r1, skip, row0=x.C, rows=skip.C)
        segs.append(ops)
        # ---- encoder, last block first; one segment per resnet layer
        ops = []
        nblocks_per_stage = [len(s) for s in self.stages]
        boundaries = set()
        acc = 0
        for n in nblocks_per_stage:
            acc += n
            boundaries.add(acc)
        pending = []      # identically shaped weight gradients of the current stage (see _wgrad_encoder)
        for bi in range(len(self.block_io) - 1, -1, -1):
            b, x, a1, idn, out = self.block_io[bi]
            d_r2, g_masked = self._bn_bwd(ops, b["conv2"], grad[id(out)], want_dres=True)
            if b["down"] is not None:
                # the downsample branch (BN backward, weight gradient, dgrad into a fresh grad[x]) on branch lane 1, next
                # to the conv2 -> conv1 chain; the chain's last dgrad accumulates onto it behind the join
                d_rd, _ = self._bn_bwd(ops, b["down"], g_masked, lane=BRANCH_LANE)
                ops.append(self._wgrad_op(b["down"], x, None, 0, d_rd, lane=BRANCH_LANE))
                add_grad(ops, b["down"], d_rd, x, lane=BRANCH_LANE)
            self._wgrad_encoder(ops, pending, b["conv2"], a1, d_r2)
            add_grad(ops, b["conv2"], d_r2, a1)
            d_r1, _ = self._bn_bwd(ops, b["conv1"], grad[id(a1)])
            self._wgrad_encoder(ops, pending, b["conv1"], x, d_r1)
            if b["down"] is not None:
                if BRANCH_LANE:
                    ops.append(make_op(_lib.OP_JOIN, n=BRANCH_LANE))
                add_grad(ops, b["conv1"], d_r1, x)
            else:
                assert id(x) not in grad
                gx = self._newT(x)
                grad[id(x)] = gx
                ops.append(self._dgrad_op(b["conv1"], d_r1, gx, res=g_masked))
                self._grad_producer[id(gx)] = ops[-1]
            if bi in boundaries or bi == 0:
                self._flush_wgrad_group(ops, pending)      # layer1's group overlaps the max-pool / stem backward below
            if bi in boundaries and bi != len(self.block_io):
                segs.append(ops)
                ops = []
        # ---- maxpool + stem
        g_f1 = grad[id(self.f1)]
        self._grad_producer[id(g_f1)] = None      # the max-pool backward accumulates into it after the dgrads
        ops.append(make_op(_lib.OP_MAXPOOL_BWD, dtype=self.dtype, B=B, H=self.f1.H, W=self.f1.W, C=64,
                           dy=grad[id(self.p1)].ptr, lddy=grad[id(self.p1)].ld, idx=self.pool_idx.data_ptr(),
                           dx=g_f1.ptr, lddx=g_f1.ld, accumulate=1))
        d_r, _ = self._bn_bwd(ops, self.stem, g_f1)
        if self.stem_s2d:
            # the stem's weight gradient from the same windowed rows as its forward (d3fk_wgrad_params.mode 2): TMA-fed, K = 256
            ops.append(make_op(_lib.OP_WGRAD, dtype=self.dtype, mode=2, src0=self.xs2d.data_ptr(), c0=64, c1=0, ld0=16, up0=0,
                               B=self.B, Hi=self.H // 2, Wi=self.W // 2, Ho=d_r.H, Wo=d_r.W, kh=4, kw=1, stride=1, pad=2,
                               dy=d_r.ptr, ldy=d_r.ld, Cout=d_r.C, cin_real=3, cout_real=self.stem.cout,
                               dw=self._gptr(self.stem.name + ".weight")))
        else:
            ops.append(self._wgrad_op(self.stem, self.x8, None, 0, d_r))
        self.dx_op_index = None
        if self.want_dx:
            # the input gradient: the stem's transposed convolution of d_raw, fp32 NCHW (run_backward patches out_nchw)
            f = dict(dtype=self.dtype, mode=1, src0=d_r.ptr, c0=d_r.C, ld0=d_r.ld, B=B, Hi=d_r.H, Wi=d_r.W, Ho=self.H,
                     Wo=self.W, kh=7, kw=7, stride=2, pad=3, w=self.w_dgrad[self.stem.name].data_ptr(), Cout=3, out_nchw=None)
            self.dx_op_index = len(ops)
            ops.append(make_op(_lib.OP_CONV, **f))
        segs.append(ops)
        return segs

    # ------------------------------------------------------------------ execution
    def run_pack(self, stream):
        self.pack_ops.run(stream)

    def run_pack_bucket(self, i, stream):
        if self.pack_bucket_ops[i] is not None:
            self.pack_bucket_ops[i].run(stream)

    def run_forward(self, x, y, stream):
        for i in self.in_op_indices:
            op_params(self.fwd_ops.array[i]).src = x.data_ptr()
        op_params(self.fwd_ops.array[self.out_op_index]).out_nchw = y.data_ptr()
        self.fwd_ops.run(stream)

    def run_backward(self, dy, stream, after_segment=None, dx=None):
        """Segments run back to back on `stream`; their weight-gradient kernels stay on libd3fk's side stream (no join
        between segments, so the big decoder wgrads overlap the latency-bound encoder segments).  `after_segment(i)`
        (data-parallel hook) must order its consumer behind BOTH streams; the final join orders `stream` itself.
        dx: fp32 NCHW [B,3,H,W] that receives the input gradient (want_dx plans only; required there)."""
        op_params(self.bwd_segments[0].array[self.dy_op_index]).src = dy.data_ptr()
        if self.want_dx:
            if dx is None:
                raise RuntimeError("this plan computes the input gradient: run_backward needs dx")
            op_params(self.bwd_segments[-1].array[self.dx_op_index]).out_nchw = dx.data_ptr()
        for i, seg in enumerate(self.bwd_segments):
            seg.run(stream, join=False)
            if after_segment is not None:
                after_segment(i)
        _lib.side_stream_join(stream)
