"""Bit-exact kernel tests on integer-valued operands (-m gpu), pinned to the launch classes of the benchmarked plans.

Activations, weights and gradients here are small integers (uniform over {-2..2} or {-1, 0, 1}).  Every value is then exact
in bf16 and fp32, every product is an exact small integer and every partial sum is an integer; below 2^21 in magnitude it is
exact in fp32 in ANY summation order (per-thread FFMA, tcgen05 accumulation in tensor memory, the split-K reduce-scatter, fp32
atomics).  So every convolution, dgrad and weight gradient of either engine must equal a float64 reference EXACTLY, and a
bf16 output must equal `ref64.to(torch.bfloat16)` (the kernels store with round-to-nearest-even).  Epilogues stay exact with
a power-of-two scale, an integer shift and an integer residual.  One wrong pixel, channel, border tap or k-block moves a
norm-relative error by less than 1e-2 on these tensor sizes; here it is a mismatch at a named (n, h, w, c).

Only quantities that are not integer by construction get a bound, each derived in the table below: the BatchNorm statistics
once a channel's sums exceed 2^21 (they are accumulated as per-CTA fp32 partials before the double atomics), and BatchNorm
backward, whose coefficients involve invstd.

The float64 reference is written from the semantics in include/d3fk.h with torch float64 ops (conv2d, conv_transpose2d,
conv2d_weight, nearest upsample, cat; epilogue scale -> shift -> res -> relu -> stats), independently of op_interpreter.py.

Launch classes: with D3FK_VERBOSE=1 the library prints one `[d3fk] conv<..> / slab<..> / wgrad<..> / wgrad_slab<..>` line per
launch.  Every case declares the class(es) it must hit and the test asserts them, so a changed path-selection threshold cannot
silently move a case onto another kernel.  test_benchmarked_plans_only_launch_pinned_classes runs the benchmarked plans and
asserts that every class they launch is one a case here pins."""
import os
import re

import pytest
import torch
import torch.nn.functional as F

from denoising_diffusion_deep_fake_b200 import _lib
from test_gpu_ops import BW_CASES, CONV_BN_CASES, CONV_CASES, HEAD_CASES, WGRAD_CASES, WGRAD_GROUP_CASES

DEV = "cuda:0"
F32, BF16 = _lib.F32, _lib.BF16
DTYPES = [F32, BF16]
TDT = {F32: torch.float32, BF16: torch.bfloat16}

# ---- constants (each fixed from first principles, none fitted to observed errors) ----
EXACT_LIMIT = 2 ** 21    # |integer partial sum| below this is exact in fp32 (24-bit significand) with 3 bits to spare
U = 2.0 ** -24           # fp32 unit roundoff: one rounding of a value v errs by at most U * |v|
BF16_REL = 2.0 ** -8     # bf16 store: RNE errs by half an ulp = 2^-9 relative; doubled for the fp32 terms it rounds
BN_BWD_FP32_OPS = 16     # fp32 roundings on the BN-backward apply chain (A, Bm, C1: 6; x - mean, two fmaf: 3; slack to 2^4)
XHAT_OPS = 3             # per term of sum(g' * xhat): x - mean, * invstd, * g' — three roundings before the summation
SCALES = (0.5, 1.0, 2.0)  # epilogue scale: powers of two keep v * scale exact
SHIFT_MAX = 4            # epilogue shift / bias: integers in [-4, 4]
RES_MAX = 2              # residual: integers in [-2, 2]
VALUE_SETS = ((2, 2), (2, 1), (1, 1))   # (max |activation|, max |weight or dY|), narrowed in this order until the budget holds


def _out_hw(c):
    if c.get("mode", 0) == 1:
        return c["Hi"] * c["stride"], c["Wi"] * c["stride"]
    return (c["Hi"] + 2 * c["pad"] - c["k"]) // c["stride"] + 1, (c["Wi"] + 2 * c["pad"] - c["k"]) // c["stride"] + 1


def budget(kind, c, amax, wmax):
    """Largest |partial sum| (and |epilogue value|) the case can produce with operands bounded by amax / wmax."""
    if kind == "conv":                                   # K terms per output: kh * kw * input channels
        acc = c["k"] * c["k"] * (c["c0"] + c.get("c1", 0)) * amax * wmax
        v = acc * (max(SCALES) if c.get("affine") else 1) + (SHIFT_MAX if c.get("affine") or c.get("bias") else 0)
        return v + (RES_MAX if c.get("res") else 0)
    if kind == "wgrad":                                  # M terms per weight: every output pixel of the batch
        Ho, Wo = _out_hw(c)
        return c["B"] * Ho * Wo * amax * wmax + c.get("dw0", 0)
    raise ValueError(kind)


def value_set(kind, c):
    for amax, wmax in VALUE_SETS:
        if budget(kind, c, amax, wmax) <= EXACT_LIMIT:
            return amax, wmax
    raise AssertionError(f"{kind} case {c}: no value set keeps the partial sums below 2^21")


def _ints(shape, vmax, g):
    return torch.randint(-vmax, vmax + 1, shape, generator=g).float()


def exact_operands(kind, c, seed):
    """Integer-valued operands of a conv / wgrad case, value set narrowed to the 2^21 budget (CPU fp32 tensors)."""
    g = torch.Generator().manual_seed(seed)
    amax, wmax = c.get("vals") or value_set(kind, c)
    B, Hi, Wi, c0, c1, up0 = c["B"], c["Hi"], c["Wi"], c["c0"], c.get("c1", 0), c.get("up0", 0)
    Ho, Wo = _out_hw(c)
    t = {"src0": _ints((B, Hi >> up0, Wi >> up0, c0), amax, g)}
    if c1:
        t["src1"] = _ints((B, Hi, Wi, c1), amax, g)
    if kind == "wgrad":
        t["dy"] = _ints((B, Ho, Wo, c["Cout"]), wmax, g)
        return t
    t["w"] = _ints((c["Cout"], c["k"] * c["k"] * (c0 + c1)), wmax, g)
    if c.get("res"):
        t["res"] = _ints((B, Ho, Wo, c["Cout"]), RES_MAX, g)
    if c.get("affine"):
        t["scale"] = torch.tensor(SCALES)[torch.randint(0, len(SCALES), (c["Cout"],), generator=g)]
    if c.get("affine") or c.get("bias"):
        t["shift"] = _ints((c["Cout"],), SHIFT_MAX, g)
    if c.get("bw") is not None:
        t["bw_x"] = _ints((B, Ho, Wo, c["Cout"]), 3, g)
        t["bw_act"] = _ints((B, Ho, Wo, c["Cout"]), 2, g).clamp_min(0)
        t["bw_mean"] = torch.randn(c["Cout"], generator=g) * 0.3
        t["bw_invstd"] = torch.rand(c["Cout"], generator=g) + 0.5
    return t


# ---- float64 reference (include/d3fk.h semantics) ----
def ref_gather(src0, src1, up0):
    a = src0
    if up0:
        a = a.repeat_interleave(2, 1).repeat_interleave(2, 2)
    if src1 is not None:
        a = torch.cat([a, src1], 3)
    return a.permute(0, 3, 1, 2)


def ref_conv_acc(t, c):
    """Accumulator of a mode-0 / mode-1 convolution, NHWC float64."""
    k, s, p, Cout = c["k"], c["stride"], c["pad"], c["Cout"]
    A = ref_gather(t["src0"].double(), t["src1"].double() if "src1" in t else None, c.get("up0", 0))
    w = t["w"].double().view(Cout, k, k, -1)
    if c.get("mode", 0) == 0:
        out = F.conv2d(A, w.permute(0, 3, 1, 2), stride=s, padding=p)
    else:
        Ho, Wo = _out_hw(c)
        opad = (Ho - ((c["Hi"] - 1) * s - 2 * p + k), Wo - ((c["Wi"] - 1) * s - 2 * p + k))
        out = F.conv_transpose2d(A, w.permute(3, 0, 1, 2), stride=s, padding=p, output_padding=opad)
    return out.permute(0, 2, 3, 1)


def ref_epilogue(acc, t, c):
    v = acc
    if "scale" in t:
        v = v * t["scale"].double() + t["shift"].double()
    elif "shift" in t:
        v = v + t["shift"].double()
    if "res" in t:
        v = v + t["res"].double()
    if c.get("relu"):
        v = v.clamp_min(0)
    return v


def ref_wgrad(x, dy, c):
    """dW[co][ci][kh][kw] (OIHW) of a mode-0 convolution, float64."""
    A = ref_gather(x["src0"].double(), x["src1"].double() if "src1" in x else None, c.get("up0", 0))
    return torch.nn.grad.conv2d_weight(A, (c["Cout"], A.shape[1], c["k"], c["k"]), dy.double().permute(0, 3, 1, 2),
                                       stride=c["stride"], padding=c["pad"])


# ---- comparisons ----
def assert_equal(got, ref, what, names="nhwc"):
    """Bit-exact comparison; on a mismatch: the count and the first differing indices (no norm)."""
    ref = ref.to(got.dtype)
    if torch.equal(got, ref):
        return
    bad = got != ref
    idx = tuple(bad.nonzero()[0].tolist())
    raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} values differ; first at "
                         f"({', '.join(f'{n}={i}' for n, i in zip(names, idx))}): got {got[idx].item()} want {ref[idx].item()}")


def assert_within(got, ref, bound, what, names="nhwc"):
    err = (got.double() - ref.double()).abs()
    bad = err > bound
    if bad.any():
        idx = tuple(bad.nonzero()[0].tolist())
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} values outside the bound; first at "
                             f"({', '.join(f'{n}={i}' for n, i in zip(names, idx))}): got {got[idx].item()} want "
                             f"{ref[idx].item()} bound {bound[idx].item() if torch.is_tensor(bound) else bound}")


def check_stats(got, v, what):
    """got [2][C] double (sum, sumsq of the fp32 epilogue value v).  Per channel: EXACT where the channel's sum of |terms|
    is <= 2^21 (every fp32 partial is then an exact integer), otherwise |err| <= M * U * sum|terms| (recursive summation of
    at most M = B*H*W terms, rounded products included).  Returns the check applied to each row."""
    v = v.reshape(-1, v.shape[-1]).double()
    M = v.shape[0]
    applied = []
    for row, terms in ((0, v), (1, v * v)):
        ref, mag = terms.sum(0), terms.abs().sum(0)
        exact = mag <= EXACT_LIMIT
        if exact.any():
            assert_equal(got[row][exact], ref[exact], f"{what} stats[{row}] (exact: sum of |terms| <= 2^21)", "c")
        if (~exact).any():
            assert_within(got[row][~exact], ref[~exact], M * U * mag[~exact], f"{what} stats[{row}] (fp32-partial bound)", "c")
        applied.append("exact" if exact.all() else "bound" if not exact.any() else "mixed")
    return applied


# ---- launch classes (the D3FK_VERBOSE=1 lines) ----
_RX = [
    (re.compile(r"\[d3fk\] conv<(\d+),(\d+)> mode=(\d+) .* KS=(\d+) .* epi=(\d+)"),
     lambda m: f"conv<{m[1]},{m[2]}> mode={m[3]} KS{'>1' if int(m[4]) > 1 else '=1'} epi={m[5]}"),
    (re.compile(r"\[d3fk\] slab<(\d+)> mode=(\d+) M=\d+ C=(\d+) .* S=(\d+) .* flat=(\d+) RT=-?\d+ epi=(\d+)"),
     lambda m: f"slab<{m[1]}> mode={m[2]} C={m[3]} S{'>1' if int(m[4]) > 1 else '=1'} flat={m[5]} epi={m[6]}"),
    (re.compile(r"\[d3fk\] wgrad<(\d+)> .* group=(\d+) .* cl=(\d+) splits=(\d+) .* tma=(\d+)"),
     lambda m: f"wgrad<{m[1]}> tma={m[5]} cl{'>1' if int(m[3]) > 1 else '=1'} splits{'>1' if int(m[4]) > 1 else '=1'} "
               f"group{'>1' if int(m[2]) > 1 else '=1'}"),
    (re.compile(r"\[d3fk\] wgrad_slab<(\d+)> M=\d+ C=(\d+) W=\d+ S=(\d+)"),
     lambda m: f"wgrad_slab<{m[1]}> C={m[2]} S{'>1' if int(m[3]) > 1 else '=1'}"),
]


def launched_classes(err_text):
    out = []
    for line in err_text.splitlines():
        if not line.startswith("[d3fk] "):
            continue
        for rx, fmt in _RX:
            m = rx.search(line)
            if m:
                out.append(fmt(m))
                break
        else:
            if re.match(r"\[d3fk\] (conv|slab|wgrad|wgrad_slab)<", line):
                raise AssertionError(f"unparsed launch line: {line}")
    return out


def op_classes(op):
    """Classes of the kernels that print no launch line, derived from the op record as their launchers dispatch on it."""
    p = _lib.op_params(op)
    dt = {F32: "f32", BF16: "bf16"}.get(getattr(p, "dtype", -1), "?")
    k = op.kind
    if k in (_lib.OP_BN_BWD, _lib.OP_BN_BWD_APPLY):
        xm = int(bool(p.relu and p.mask_from_x))
        return ([f"bn_bwd_reduce<{dt}> xmask={xm}"] if k == _lib.OP_BN_BWD else []) + [f"bn_bwd_apply<{dt}> xmask={xm}"]
    if k == _lib.OP_NCHW2NHWC:
        return [f"nchw2nhwc<{dt}> chansum={int(bool(p.chansum))}"]
    if (k == _lib.OP_CONV and p.dtype == BF16 and p.mode == 0 and p.kh == 3 and p.kw == 3 and p.stride == 1 and p.pad == 1
            and p.c0 == 16 and p.c1 == 0 and p.up0 == 0 and 1 <= p.Cout <= 3 and p.out_nchw and not p.out and not p.res
            and not p.stats and not p.relu and not p.scale and not p.bw_x and p.Ho == p.Hi and p.Wo == p.Wi
            and p.Hi % 32 == 0 and p.Wi % 32 == 0 and p.ld0 % 8 == 0):        # try_launch_head_conv's conditions
        return [f"head_conv<{128 if p.Wi % 128 == 0 else 64 if p.Wi % 64 == 0 else 32}>"]
    return []


@pytest.fixture(scope="module")
def verbose():
    """D3FK_VERBOSE=1 for this module: tc_init re-reads it on every d3fk_init (the raw export; _lib.init caches)."""
    lib = _lib.load()
    os.environ["D3FK_VERBOSE"] = "1"
    assert lib.d3fk_init(0) == 0, lib.d3fk_last_error()
    _lib.init(0)
    yield
    os.environ["D3FK_VERBOSE"] = "0"
    lib.d3fk_init(0)


def assert_pinned(capfd, declared, extra=()):
    seen = set(launched_classes(capfd.readouterr().err)) | set(extra)
    print("PIN", sorted(seen))
    missing = set(declared) - seen
    assert not missing, f"declared launch class(es) {sorted(missing)} not launched; launched: {sorted(seen)}"
    stray = seen - set(declared)
    assert not stray, f"launched class(es) {sorted(stray)} the case does not declare"


def run(op):
    _lib.run_single(op, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert _lib.load().d3fk_device_error_flag() == 0, "kernel watchdog tripped"


def dev(t, dtype=None):
    return t.to(DEV) if dtype is None else t.to(DEV).to(dtype)


# ---- declared launch classes of the cases (bf16 engine; the fp32 engine is the FFMA kernel and prints none) ----
PIN_CONV = {
    0: {'slab<64> mode=0 C=64 S=1 flat=0 epi=0'}, 1: {'conv<128,2> mode=0 KS>1 epi=3'}, 2: {'conv<128,0> mode=0 KS>1 epi=0'},
    3: {'conv<128,0> mode=0 KS=1 epi=0'}, 4: {'conv<64,0> mode=0 KS=1 epi=0'}, 5: {'conv<128,1> mode=0 KS>1 epi=0'},
    6: {'conv<32,1> mode=0 KS=1 epi=3'}, 7: {'conv<16,1> mode=0 KS=1 epi=0'}, 8: {'head_conv<32>'},
    9: {'conv<128,2> mode=0 KS>1 epi=0'}, 10: {'slab<16> mode=0 C=16 S>1 flat=0 epi=0'}, 11: {'conv<128,2> mode=0 KS>1 epi=0'},
    12: {'conv<128,2> mode=0 KS>1 epi=3'}, 13: {'conv<128,1> mode=0 KS>1 epi=0'}, 14: {'conv<128,1> mode=1 KS>1 epi=0'},
    15: {'slab<16> mode=0 C=16 S>1 flat=0 epi=0'}, 16: {'slab<64> mode=1 C=64 S=1 flat=0 epi=0'},
    17: {'conv<64,1> mode=1 KS=1 epi=0'}, 18: {'conv<64,1> mode=1 KS=1 epi=0'}, 19: {'conv<16,0> mode=1 KS=1 epi=0'},
    20: {'slab<32> mode=0 C=32 S>1 flat=0 epi=0'}, 21: {'slab<32> mode=1 C=32 S>1 flat=0 epi=0'},
    22: {'slab<64> mode=1 C=32 S>1 flat=0 epi=0'}, 23: {'slab<32> mode=1 C=16 S>1 flat=0 epi=0'},
    24: {'slab<16> mode=0 C=16 S>1 flat=0 epi=3'}, 25: {'conv<128,2> mode=1 KS>1 epi=0'},
    26: {'slab<64> mode=0 C=64 S=1 flat=0 epi=0'}, 27: {'slab<64> mode=0 C=64 S=1 flat=0 epi=0'},
    28: {'slab<16> mode=0 C=16 S=1 flat=0 epi=0'}, 29: {'slab<32> mode=0 C=32 S>1 flat=0 epi=0'}, 30: {'head_conv<64>'},
    31: {'slab<16> mode=0 C=16 S>1 flat=0 epi=0'}, 32: {'slab<32> mode=1 C=32 S>1 flat=0 epi=0'},
    33: {'slab<16> mode=0 C=16 S>1 flat=0 epi=0'}, 34: {'slab<16> mode=1 C=16 S>1 flat=0 epi=0'},
    35: {'slab<32> mode=0 C=128 S=1 flat=0 epi=0'}, 36: {'conv<64,2> mode=0 KS=1 epi=3'},
    37: {'slab<32> mode=0 C=128 S=1 flat=0 epi=0'}
}
PIN_WGRAD = {
    0: {'wgrad<64> tma=1 cl=1 splits>1 group=1'}, 1: {'wgrad<128> tma=0 cl=1 splits=1 group=1'},
    2: {'wgrad<128> tma=0 cl=1 splits>1 group=1'}, 3: {'wgrad<64> tma=0 cl>1 splits>1 group=1'},
    4: {'wgrad<128> tma=0 cl=1 splits=1 group=1'}, 5: {'wgrad<64> tma=0 cl=1 splits>1 group=1'},
    6: {'wgrad<64> tma=0 cl=1 splits>1 group=1'}, 7: {'wgrad<128> tma=1 cl=1 splits=1 group=1'},
    8: {'wgrad<64> tma=0 cl=1 splits>1 group=1'}, 9: {'wgrad_slab<16> C=16 S>1'}, 10: {'wgrad_slab<16> C=16 S>1'},
    11: {'wgrad_slab<32> C=32 S>1'}, 12: {'wgrad_slab<32> C=64 S=1'}, 13: {'wgrad_slab<32> C=16 S>1'},
    14: {'wgrad_slab<16> C=64 S=1'}
}
PIN_BW = {
    0: {'conv<128,2> mode=1 KS>1 epi=2'}, 1: {'conv<128,2> mode=1 KS>1 epi=2'}, 2: {'conv<128,2> mode=1 KS>1 epi=2'},
    3: {'conv<64,1> mode=1 KS=1 epi=2'}, 4: {'slab<64> mode=1 C=64 S=1 flat=0 epi=2'},
    5: {'slab<32> mode=1 C=32 S>1 flat=0 epi=2'}, 6: {'slab<16> mode=1 C=16 S>1 flat=0 epi=2'},
    7: {'slab<32> mode=1 C=16 S>1 flat=0 epi=2'}
}
PIN_CONV_BN = {
    0: {'conv<128,2> mode=0 KS>1 epi=1'}, 1: {'conv<128,2> mode=0 KS>1 epi=1'}, 2: {'conv<128,2> mode=0 KS>1 epi=1'},
    3: {'conv<128,2> mode=0 KS>1 epi=1'}, 4: {'conv<128,0> mode=0 KS>1 epi=1'}, 5: {'conv<128,0> mode=0 KS=1 epi=1'},
    6: {'conv<128,1> mode=0 KS>1 epi=1'}, 7: {'slab<64> mode=0 C=64 S=1 flat=0 epi=0'}
}
PIN_GROUP = {
    0: {'wgrad<64> tma=0 cl>1 splits>1 group>1'}, 1: {'wgrad<128> tma=0 cl=1 splits=1 group>1'},
    2: {'wgrad<128> tma=0 cl=1 splits=1 group>1'}, 3: {'wgrad<128> tma=0 cl=1 splits=1 group>1'},
    4: {'wgrad<128> tma=0 cl=1 splits=1 group=1'}, 5: {'wgrad<64> tma=0 cl=1 splits=1 group>1'},
    6: {'wgrad<128> tma=0 cl>1 splits>1 group>1'}
}
PIN_HEAD = {
    (0, False): {'head_conv<64>'}, (0, True): {'head_conv<64>'}, (1, False): {'head_conv<128>'}, (1, True): {'head_conv<128>'},
    (2, False): {'head_conv<32>'}, (2, True): {'head_conv<32>'}, (3, False): {'head_conv<32>'}, (3, True): {'head_conv<32>'},
    (4, False): {'head_conv<128>'}, (4, True): {'head_conv<128>'}, (5, False): {'slab<16> mode=0 C=16 S>1 flat=0 epi=0'},
    (5, True): {'slab<16> mode=0 C=16 S>1 flat=0 epi=3'}
}

# forms the benchmarked plans launch that no case above reaches: eval-affine epilogues (FUSE 3) of the generic and slab
# paths, unsplit 128-wide tiles (> 74 output tiles), 32-wide TMA tiles, the decoder tail at 128 x 128, deep clustered wgrads
PLAN_CONV_CASES = [
    dict(B=2, Hi=16, Wi=16, c0=64, c1=0, up0=0, Cout=128, k=3, stride=2, pad=1, mode=0, relu=1, affine=True,
         pin={"conv<128,0> mode=0 KS>1 epi=3"}),
    dict(B=2, Hi=16, Wi=16, c0=64, c1=0, up0=0, Cout=128, k=1, stride=2, pad=0, mode=0, affine=True,
         pin={"conv<128,0> mode=0 KS=1 epi=3"}),
    dict(B=160, Hi=8, Wi=8, c0=128, c1=0, up0=0, Cout=128, k=3, stride=1, pad=1, mode=0, relu=1, res=True, affine=True,
         pin={"conv<128,2> mode=0 KS=1 epi=3"}),
    dict(B=160, Hi=8, Wi=8, c0=128, c1=0, up0=0, Cout=128, k=3, stride=1, pad=1, mode=1, res=True,
         pin={"conv<128,2> mode=1 KS=1 epi=0"}),
    dict(B=48, Hi=8, Wi=8, c0=256, c1=0, up0=0, Cout=128, k=3, stride=2, pad=1, mode=1, pin={"conv<128,1> mode=1 KS=1 epi=0"}),
    dict(B=2, Hi=64, Wi=64, c0=128, c1=0, up0=0, Cout=32, k=3, stride=1, pad=1, mode=0, stats=True,
         pin={"conv<32,2> mode=0 KS=1 epi=0"}),
    dict(B=2, Hi=64, Wi=64, c0=128, c1=0, up0=0, Cout=32, k=3, stride=1, pad=1, mode=0, relu=1, affine=True,
         pin={"conv<32,2> mode=0 KS=1 epi=3"}),
    dict(B=2, Hi=128, Wi=128, c0=32, c1=0, up0=0, Cout=16, k=3, stride=1, pad=1, mode=0, stats=True,
         pin={"slab<16> mode=0 C=32 S>1 flat=0 epi=0"}),
    dict(B=2, Hi=128, Wi=128, c0=32, c1=0, up0=0, Cout=16, k=3, stride=1, pad=1, mode=0, relu=1, affine=True,
         pin={"slab<16> mode=0 C=32 S>1 flat=0 epi=3"}),
    dict(B=3, Hi=32, Wi=32, c0=32, c1=0, up0=0, Cout=32, k=3, stride=1, pad=1, mode=0, relu=1, affine=True,
         pin={"slab<32> mode=0 C=32 S>1 flat=0 epi=3"}),
    dict(B=2, Hi=16, Wi=16, c0=64, c1=0, up0=0, Cout=64, k=3, stride=1, pad=1, mode=0, relu=1, affine=True,
         pin={"slab<64> mode=0 C=64 S=1 flat=0 epi=3"}),
]
PLAN_WGRAD_CASES = [
    dict(B=256, Hi=8, Wi=8, c0=128, c1=0, up0=0, Cout=128, k=3, stride=1, pad=1, pin={"wgrad<128> tma=1 cl>1 splits>1 group=1"}),
    dict(B=256, Hi=4, Wi=4, c0=256, c1=0, up0=0, Cout=512, k=3, stride=2, pad=1, pin={"wgrad<128> tma=0 cl>1 splits>1 group=1"}),
    dict(B=5, Hi=128, Wi=128, c0=32, c1=0, up0=0, Cout=16, k=3, stride=1, pad=1, pin={"wgrad_slab<16> C=32 S>1"}),
]
PLAN_CONV_BN_CASES = [    # > 74 output tiles, all resident: fused without split K
    dict(B=160, Hi=8, Wi=8, c0=128, c1=0, up0=0, Cout=128, k=3, stride=1, pad=1, relu=1, res=True,
         pin={"conv<128,2> mode=0 KS=1 epi=1"}),
]
CONV_ALL = [(f"CONV_CASES[{i}]", c, PIN_CONV[i]) for i, c in enumerate(CONV_CASES)] + \
           [(f"PLAN_CONV_CASES[{i}]", c, c["pin"]) for i, c in enumerate(PLAN_CONV_CASES)]
WGRAD_ALL = [(f"WGRAD_CASES[{i}]", c, PIN_WGRAD[i]) for i, c in enumerate(WGRAD_CASES)] + \
            [(f"PLAN_WGRAD_CASES[{i}]", c, c["pin"]) for i, c in enumerate(PLAN_WGRAD_CASES)]
CONV_BN_ALL = [(f"CONV_BN_CASES[{i}]", c, PIN_CONV_BN[i]) for i, c in enumerate(CONV_BN_CASES)] + \
              [(f"PLAN_CONV_BN_CASES[{i}]", c, c["pin"]) for i, c in enumerate(PLAN_CONV_BN_CASES)]


# ---- cases added for the forms only the plans launch ----
STEM_PIN = {"conv<64,2> mode=0 KS=1 epi=0", "wgrad<64> tma=1 cl>1 splits>1 group=1"}
STEM_CASES = [dict(B=2, H=64, W=64), dict(B=3, H=128, W=128), dict(B=1, H=256, W=64)]
INPLACE_CASES = [
    # add_grad into an existing gradient (res == out): the stride-2 conv1 of a stage's first block, generic and split-K
    dict(B=4, Hi=8, Wi=8, c0=128, Cout=64, k=3, stride=2, pad=1, mode=1, pin={"conv<64,1> mode=1 KS=1 epi=0"}),
    dict(B=4, Hi=4, Wi=4, c0=256, Cout=128, k=3, stride=2, pad=1, mode=1, pin={"conv<128,1> mode=1 KS>1 epi=0"}),
    dict(B=16, Hi=4, Wi=4, c0=256, Cout=256, k=3, stride=1, pad=1, mode=1, pin={"conv<128,2> mode=1 KS>1 epi=0"}),
    dict(B=3, Hi=32, Wi=32, c0=32, Cout=32, k=3, stride=1, pad=1, mode=1, pin={"slab<32> mode=1 C=32 S>1 flat=0 epi=0"}),
]
SLICED_CASES = [
    # decoder conv1 dgrad split at the upsample / skip boundary: weight pointer offset by row0, Cout = rows
    dict(B=160, Hi=8, Wi=8, c0=128, cin=384, row0=256, rows=128, k=3, stride=1, pad=1, mode=1, pin={"conv<128,2> mode=1 KS=1 epi=0"}),
    dict(B=2, Hi=8, Wi=8, c0=128, cin=384, row0=0, rows=256, k=3, stride=1, pad=1, mode=1, pin={"conv<128,2> mode=1 KS>1 epi=0"}),
    dict(B=2, Hi=32, Wi=32, c0=32, cin=128, row0=64, rows=64, k=3, stride=1, pad=1, mode=1, pin={"slab<64> mode=1 C=32 S>1 flat=0 epi=0"}),
]
HALVES_CASES = [dict(B=76, Hi=32, Wi=32, c0=64, Cout=32, k=3, stride=1, pad=1, cin=128, dw0=3, pin={"wgrad_slab<32> C=64 S=1"})]
CHANSUM_CASES = [dict(B=2, H=64, W=64), dict(B=3, H=32, W=96)]
BN_BWD_CASES = [(64, 2 * 16 * 16), (16, 3 * 64 * 64), (256, 1000), (32, 50000), (512, 8)]


def all_budget_cases():
    """Every (kind, case) of this file whose operands exact_operands draws."""
    out = [("conv", c) for _, c, _ in CONV_ALL] + [("conv", c) for c in BW_CASES] + [("wgrad", c) for _, c, _ in WGRAD_ALL]
    out += [("conv", dict(c, mode=0, vals=(1, 1))) for _, c, _ in CONV_BN_ALL]
    out += [("conv", dict(c0=16, c1=0, up0=0, k=3, stride=1, pad=1, mode=0, nchw=True, bias=True, **c)) for c in HEAD_CASES]
    out += [("wgrad", dict(B=B, Hi=H, Wi=H, c0=C, Cout=C, k=3, stride=1, pad=1)) for _, B, H, C in WGRAD_GROUP_CASES]
    out += [("conv", dict(c, res=True)) for c in INPLACE_CASES] + [("conv", dict(c, res=True, bw=1)) for c in INPLACE_CASES]
    out += [("conv", dict(c, Cout=c["rows"])) for c in SLICED_CASES]
    out += [("wgrad", dict(c, c0=c["cin"])) for c in HALVES_CASES]
    for s in STEM_CASES:                                # forward K = 7*7*3; weight gradient M = B*H/2*W/2
        out += [("conv", dict(B=s["B"], Hi=s["H"], Wi=s["W"], c0=3, Cout=64, k=7, stride=2, pad=3)),
                ("wgrad", dict(B=s["B"], Hi=s["H"], Wi=s["W"], c0=3, Cout=64, k=7, stride=2, pad=3))]
    return out


def test_exact_budget():
    """Every case of this file keeps its largest |partial sum| at or below 2^21 with the value set it draws from."""
    cases = all_budget_cases()
    assert len(cases) == len(CONV_ALL) + len(BW_CASES) + len(WGRAD_ALL) + len(CONV_BN_ALL) + len(HEAD_CASES) + \
        len(WGRAD_GROUP_CASES) + 2 * len(INPLACE_CASES) + len(SLICED_CASES) + len(HALVES_CASES) + 2 * len(STEM_CASES)
    for kind, c in cases:
        amax, wmax = c.get("vals") or value_set(kind, c)
        assert budget(kind, c, amax, wmax) <= EXACT_LIMIT, (kind, c)


def test_budget_narrows_long_reductions():
    """The generator narrows the value set for long reductions instead of overflowing the budget."""
    assert value_set("conv", dict(k=3, c0=512, Cout=512, B=1, Hi=2, Wi=2, stride=1, pad=1)) == (2, 2)
    long = dict(B=300, Hi=64, Wi=64, c0=16, Cout=16, k=3, stride=1, pad=1)       # 1.2 M pixels of reduction
    assert value_set("wgrad", long) == (1, 1)
    with pytest.raises(AssertionError):
        value_set("wgrad", dict(long, B=600))


# ------------------------------------------------------------------ convolution / dgrad (both engines)
def conv_fields(dtype, c, g, o):
    Ho, Wo = _out_hw(c)
    f = dict(dtype=dtype, mode=c.get("mode", 0), src0=g["src0"].data_ptr(), c0=c["c0"], c1=c.get("c1", 0), ld0=c["c0"],
             ld1=c.get("c1", 0), up0=c.get("up0", 0), B=c["B"], Hi=c["Hi"], Wi=c["Wi"], Ho=Ho, Wo=Wo, kh=c["k"], kw=c["k"],
             stride=c["stride"], pad=c["pad"], w=g["w"].data_ptr(), Cout=c["Cout"], relu=c.get("relu", 0))
    if "src1" in g:
        f["src1"] = g["src1"].data_ptr()
    if c.get("nchw"):
        f["out_nchw"] = o["out"].data_ptr()
    else:
        f.update(out=o["out"].data_ptr(), ldo=c["Cout"])
    if "res" in g:
        f.update(res=g["res"].data_ptr(), ldr=c["Cout"])
    if "scale" in g:
        f["scale"] = g["scale"].data_ptr()
    if "shift" in g:
        f["shift"] = g["shift"].data_ptr()
    if "stats" in o:
        f["stats"] = o["stats"].data_ptr()
    if "bw_x" in g:
        f.update(bw_x=g["bw_x"].data_ptr(), bw_act=g["bw_act"].data_ptr(), bw_mean=g["bw_mean"].data_ptr(),
                 bw_invstd=g["bw_invstd"].data_ptr(), bw_ldx=c["Cout"], bw_ldact=c["Cout"], bw_relu=c["bw"])
    return f


_F32_FIELDS = ("scale", "shift", "bw_mean", "bw_invstd")


def run_conv_case(dtype, c, seed=0):
    """Launch one integer-valued conv case; returns (operands on the GPU, outputs, exact fp32 epilogue value v)."""
    t = exact_operands("conv", c, seed)
    g = {n: dev(v) if n in _F32_FIELDS else dev(v, TDT[dtype]) for n, v in t.items()}
    Ho, Wo = _out_hw(c)
    o = {"out": torch.zeros(c["B"], c["Cout"], Ho, Wo, device=DEV) if c.get("nchw")
         else torch.zeros(c["B"], Ho, Wo, c["Cout"], device=DEV, dtype=TDT[dtype])}
    if c.get("stats") or c.get("bw") is not None:
        o["stats"] = torch.zeros(2, c["Cout"], dtype=torch.float64, device=DEV)
    run(_lib.make_op(_lib.OP_CONV, **conv_fields(dtype, c, g, o)))
    v = ref_epilogue(ref_conv_acc(g, c), g, c)
    return g, o, v


def check_conv_outputs(c, g, o, v, what):
    if c.get("nchw"):
        assert_equal(o["out"], v.permute(0, 3, 1, 2), what + " out_nchw", "nchw")
    else:
        assert_equal(o["out"], v, what + " out")
    if c.get("bw") is not None:
        gp = v * (g["bw_act"].double() > 0) if c["bw"] else v
        xhat = (g["bw_x"].double() - g["bw_mean"].double()) * g["bw_invstd"].double()
        check_bn_bwd_sums(o["stats"], gp, xhat, what)
    elif c.get("stats"):
        check_stats(o["stats"], v, what)


def check_bn_bwd_sums(got, gp, xhat, what):
    """BN-backward sums [sum g', sum g' * xhat]: the first is a sum of integers (exact under the budget, else the
    fp32-partial bound), the second carries xhat's roundings: |err| <= (M + XHAT_OPS) * U * sum|g' * xhat|."""
    gp, xhat = gp.reshape(-1, gp.shape[-1]).double(), xhat.reshape(-1, xhat.shape[-1]).double()
    M = gp.shape[0]
    s1, a1 = gp.sum(0), gp.abs().sum(0)
    ex = a1 <= EXACT_LIMIT
    assert_equal(got[0][ex], s1[ex], f"{what} sum(g') (exact)", "c")
    assert_within(got[0][~ex], s1[~ex], M * U * a1[~ex], f"{what} sum(g') (fp32-partial bound)", "c")
    t = gp * xhat
    assert_within(got[1], t.sum(0), (M + XHAT_OPS) * U * t.abs().sum(0), f"{what} sum(g' * xhat) (bound)", "c")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("i", range(len(CONV_ALL)))
def test_conv_exact(verbose, capfd, dtype, i):
    name, c, pin = CONV_ALL[i]
    g, o, v = run_conv_case(dtype, c, seed=c.get("seed", 0) + 100 * i)
    check_conv_outputs(c, g, o, v, name)
    if dtype == BF16:
        head = op_classes(_lib.make_op(_lib.OP_CONV, **conv_fields(dtype, c, g, o)))
        assert_pinned(capfd, pin, head)


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(BW_CASES)))
def test_dgrad_bn_backward_sums_exact(verbose, capfd, i):
    c = BW_CASES[i]
    g, o, v = run_conv_case(BF16, c, seed=200 + i)
    check_conv_outputs(c, g, o, v, f"BW_CASES[{i}]")
    assert_pinned(capfd, PIN_BW[i])


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(HEAD_CASES)))
@pytest.mark.parametrize("bias", [False, True])
def test_head_conv_exact(verbose, capfd, i, bias):
    """Segmentation head (head_conv.cu, mma.sync) on integer data, every tile width; it prints no launch line."""
    c = dict(c0=16, c1=0, up0=0, k=3, stride=1, pad=1, mode=0, nchw=True, bias=bias, **HEAD_CASES[i])
    g, o, v = run_conv_case(BF16, c, seed=300 + i)
    check_conv_outputs(c, g, o, v, f"HEAD_CASES[{i}]")
    cls = op_classes(_lib.make_op(_lib.OP_CONV, **conv_fields(BF16, c, g, o)))
    assert_pinned(capfd, PIN_HEAD[(i, bias)], cls)


# ------------------------------------------------------------------ weight gradients
def wgrad_fields(dtype, c, g, dw, cin_real=None, cout_real=None):
    Ho, Wo = _out_hw(c)
    ctot = c["c0"] + c.get("c1", 0)
    f = dict(dtype=dtype, src0=g["src0"].data_ptr(), c0=c["c0"], c1=c.get("c1", 0), ld0=c["c0"], ld1=c.get("c1", 0),
             up0=c.get("up0", 0), B=c["B"], Hi=c["Hi"], Wi=c["Wi"], Ho=Ho, Wo=Wo, kh=c["k"], kw=c["k"], stride=c["stride"],
             pad=c["pad"], dy=g["dy"].data_ptr(), ldy=c["Cout"], Cout=c["Cout"], cin_real=cin_real or ctot,
             cout_real=cout_real or c["Cout"], dw=dw.data_ptr())
    if "src1" in g:
        f["src1"] = g["src1"].data_ptr()
    return f


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("i", range(len(WGRAD_ALL)))
def test_wgrad_exact(verbose, capfd, dtype, i):
    name, c, pin = WGRAD_ALL[i]
    t = exact_operands("wgrad", c, 400 + i)
    g = {n: dev(v, TDT[dtype]) for n, v in t.items()}
    cin_real, cout_real = c.get("cin_real", c["c0"] + c["c1"]), c.get("cout_real", c["Cout"])
    dw = torch.zeros(cout_real, cin_real, c["k"], c["k"], device=DEV)
    run(_lib.make_op(_lib.OP_WGRAD, **wgrad_fields(dtype, c, g, dw, cin_real, cout_real)))
    ref = ref_wgrad(g, g["dy"], c)[:cout_real, :cin_real]
    assert_equal(dw, ref, f"{name} dW", "oihw")
    if dtype == BF16:
        assert_pinned(capfd, pin)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("i", range(len(WGRAD_GROUP_CASES)))
def test_wgrad_group_exact(verbose, capfd, dtype, i):
    count, B, H, C = WGRAD_GROUP_CASES[i]
    c = dict(B=B, Hi=H, Wi=H, c0=C, Cout=C, k=3, stride=1, pad=1)
    ops = [{n: dev(v, TDT[dtype]) for n, v in exact_operands("wgrad", c, 500 + 17 * i + j).items()} for j in range(count)]
    dws = [torch.zeros(C, C, 3, 3, device=DEV) for _ in range(count)]
    base = wgrad_fields(dtype, c, ops[0], dws[0])
    for n in ("src0", "dy", "dw"):
        base.pop(n)
    run(_lib.make_op(_lib.OP_WGRAD_GROUP, base=base, count=count, src0=[o["src0"].data_ptr() for o in ops],
                     dy=[o["dy"].data_ptr() for o in ops], dw=[d.data_ptr() for d in dws]))
    for j in range(count):
        assert_equal(dws[j], ref_wgrad(ops[j], ops[j]["dy"], c), f"WGRAD_GROUP_CASES[{i}] problem {j} dW", "oihw")
    if dtype == BF16:
        assert_pinned(capfd, PIN_GROUP[i])


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(HALVES_CASES)))
def test_wgrad_halves_exact(verbose, capfd, i):
    """plan._wgrad_ops: a 128-channel input as two 64-channel halves (src0 and dW offset), accumulating into a dW that
    already holds integers (dw0)."""
    c = HALVES_CASES[i]
    cin, C = c["cin"], c["c0"]
    t = exact_operands("wgrad", dict(c, c0=cin), 600 + i)
    g = {n: dev(v, torch.bfloat16) for n, v in t.items()}
    n = c["Cout"] * cin * 9
    arena = torch.full((n + 8,), float(c["dw0"]), device=DEV)
    dw = arena[:n]
    for half in range(cin // C):
        f = wgrad_fields(BF16, c, g, dw, cin, c["Cout"])
        f.update(src0=g["src0"].data_ptr() + half * C * 2, ld0=cin, dw=dw.data_ptr() + half * C * 9 * 4)
        run(_lib.make_op(_lib.OP_WGRAD, **f))
    ref = ref_wgrad(g, g["dy"], dict(c, c0=cin)) + c["dw0"]
    assert_equal(dw.view(c["Cout"], cin, 3, 3), ref, "two-half dW", "oihw")
    assert_equal(arena[n:], torch.full((8,), float(c["dw0"]), device=DEV), "past the end of dW", "i")
    assert_pinned(capfd, c["pin"])


# ------------------------------------------------------------------ the space-to-depth stem, forward and weight gradient
@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(STEM_CASES)))
def test_stem_space_to_depth_exact(verbose, capfd, i):
    s = STEM_CASES[i]
    B, H, W = s["B"], s["H"], s["W"]
    gen = torch.Generator().manual_seed(700 + i)
    x = dev(_ints((B, 3, H, W), 2, gen))
    w = dev(_ints((64, 3, 7, 7), 2, gen))
    Hs, Ws = H // 2, W // 2
    xs = torch.zeros(B, Hs, Ws + 3, 16, device=DEV, dtype=torch.bfloat16)
    wp = torch.zeros(64, 256, device=DEV, dtype=torch.bfloat16)
    out = torch.zeros(B, Hs, Ws, 64, device=DEV, dtype=torch.bfloat16)
    st = torch.zeros(2, 64, dtype=torch.float64, device=DEV)
    conv = dict(dtype=BF16, mode=2, src0=xs.data_ptr(), c0=64, c1=0, ld0=16, ld1=0, up0=0, B=B, Hi=Hs, Wi=Ws, Ho=Hs, Wo=Ws,
                kh=4, kw=1, stride=1, pad=2, w=wp.data_ptr(), Cout=64, out=out.data_ptr(), ldo=64, stats=st.data_ptr())
    _lib.OpList([_lib.make_op(_lib.OP_NCHW2S2D, dtype=BF16, B=B, C=3, H=H, W=W, cpad=4, src=x.data_ptr(), dst=xs.data_ptr()),
                 _lib.make_op(_lib.OP_PACK_STEM, dtype=BF16, Cout=64, Cin=3, kh=7, kw=7, cin_pad=4, cout_pad=64,
                              w=w.data_ptr(), w_fwd=wp.data_ptr()),
                 _lib.make_op(_lib.OP_CONV, **conv)]).run(torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ref = F.conv2d(x.double(), w.double(), stride=2, padding=3).permute(0, 2, 3, 1)
    assert_equal(out, ref, "stem forward")
    check_stats(st, ref, "stem forward")
    dy = dev(_ints((B, Hs, Ws, 64), 2, gen), torch.bfloat16)
    dw = torch.zeros(64, 3, 7, 7, device=DEV)
    run(_lib.make_op(_lib.OP_WGRAD, dtype=BF16, mode=2, src0=xs.data_ptr(), c0=64, c1=0, ld0=16, up0=0, B=B, Hi=Hs, Wi=Ws,
                     Ho=Hs, Wo=Ws, kh=4, kw=1, stride=1, pad=2, dy=dy.data_ptr(), ldy=64, Cout=64, cin_real=3, cout_real=64,
                     dw=dw.data_ptr()))
    ref_dw = torch.nn.grad.conv2d_weight(x.double(), (64, 3, 7, 7), dy.double().permute(0, 3, 1, 2), stride=2, padding=3)
    assert_equal(dw, ref_dw, "stem weight gradient", "oihw")
    assert_pinned(capfd, STEM_PIN)


# ------------------------------------------------------------------ fused conv + BatchNorm (FUSE 1) and its two-kernel form
def ulp_bf16(x):
    e = torch.frexp(x.abs().float())[1].double()
    return torch.where(x == 0, torch.zeros_like(x, dtype=torch.float64), torch.exp2(e - 8))


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(CONV_BN_ALL)))
def test_conv_bn_exact(verbose, capfd, i):
    """Raw output exact; statistics exact or within their bound; act within one bf16 ulp (plus the fp32 rounding of the
    coefficients) of bf16(fmaf(bf16(raw), sc, sh)) [+ res, relu], sc / sh from the exact statistics in float64 -> fp32."""
    name, c, pin = CONV_BN_ALL[i]
    c = dict(c, mode=0, vals=(1, 1))
    C = c["Cout"]
    t = exact_operands("conv", dict(c, res=False), 800 + i)
    gen = torch.Generator().manual_seed(850 + i)
    Ho, Wo = _out_hw(c)
    g = {n: dev(v, torch.bfloat16) for n, v in t.items()}
    if c["res"]:
        g["res"] = dev(_ints((c["B"], Ho, Wo, C), RES_MAX, gen), torch.bfloat16)
    s = {"stats": torch.zeros(2, C, dtype=torch.float64), "gamma": torch.rand(C, generator=gen) + 0.5,
         "beta": torch.randn(C, generator=gen), "running_mean": torch.zeros(C), "running_var": torch.ones(C),
         "nbt": torch.zeros(1, dtype=torch.int64), "mean": torch.zeros(C), "invstd": torch.zeros(C), "scale": torch.zeros(C),
         "shift": torch.zeros(C), "barrier": torch.zeros(2, dtype=torch.int32)}
    s = {n: dev(v) for n, v in s.items()}
    raw = torch.zeros(c["B"], Ho, Wo, C, device=DEV, dtype=torch.bfloat16)
    act = torch.zeros_like(raw)
    conv = conv_fields(BF16, dict(c, res=False, relu=0), {n: v for n, v in g.items() if n != "res"}, {"out": raw})
    conv["stats"] = s["stats"].data_ptr()
    M = c["B"] * Ho * Wo
    bn = dict(dtype=BF16, C=C, relu=c["relu"], count=M, x=raw.data_ptr(), ldx=C, y=act.data_ptr(), ldy=C,
              stats=s["stats"].data_ptr(), gamma=s["gamma"].data_ptr(), beta=s["beta"].data_ptr(),
              running_mean=s["running_mean"].data_ptr(), running_var=s["running_var"].data_ptr(),
              num_batches_tracked=s["nbt"].data_ptr(), eps=1e-5, momentum=0.1, scale=s["scale"].data_ptr(),
              shift=s["shift"].data_ptr(), mean=s["mean"].data_ptr(), invstd=s["invstd"].data_ptr())
    if c["res"]:
        bn.update(res=g["res"].data_ptr(), ldr=C)
    run(_lib.make_op(_lib.OP_CONV_BN, conv=conv, bn=bn, barrier=s["barrier"].data_ptr()))
    v = ref_conv_acc(g, c)
    assert_equal(raw, v, f"{name} raw")
    check_stats(s["stats"], v, name)
    vf = v.reshape(-1, C)
    mean = vf.mean(0)
    var = (vf * vf).mean(0) - mean * mean
    invstd = 1.0 / torch.sqrt(var + 1e-5)
    sc = (s["gamma"].double() * invstd).float().double()
    sh = (s["beta"].double() - mean * s["gamma"].double() * invstd).float().double()
    rb = raw.double()
    y = (rb * sc + sh).float().double()
    coef_err = 4 * U * (rb.abs() * sc.abs() + sh.abs())
    if c["res"]:
        y = y + g["res"].double()
        coef_err = coef_err + 2 * U * y.abs()
    if c["relu"]:
        y = y.clamp_min(0)
    ref_act = y.to(torch.bfloat16).double()
    assert_within(act, ref_act, ulp_bf16(ref_act) + coef_err, f"{name} act (one bf16 ulp)")
    for n, ref in (("mean", mean), ("invstd", invstd), ("running_mean", 0.1 * mean),
                   ("running_var", 0.9 + 0.1 * var * M / (M - 1))):
        assert_within(s[n], ref.float(), 4 * U * ref.abs(), f"{name} {n}", "c")
    assert int(s["nbt"].item()) == 1
    assert_pinned(capfd, pin)


# ------------------------------------------------------------------ dgrad forms the plans emit
@pytest.mark.gpu
@pytest.mark.parametrize("bw", [False, True])
@pytest.mark.parametrize("i", range(len(INPLACE_CASES)))
def test_inplace_dgrad_exact(verbose, capfd, i, bw):
    """plan.add_grad into an existing gradient: res == out (the dgrad reads and overwrites the same buffer).  With bw the
    same launch carries the BN-backward sums (FUSE 2), taken over the ACCUMULATED gradient."""
    c = dict(INPLACE_CASES[i], c1=0, up0=0, res=True)
    c.pop("pin")
    if bw:
        c["bw"] = 1
    t = exact_operands("conv", c, 900 + i)
    g = {n: dev(v) if n in _F32_FIELDS else dev(v, torch.bfloat16) for n, v in t.items()}
    prior = g.pop("res")
    buf = prior.clone()
    o = {"out": buf}
    if bw:
        o["stats"] = torch.zeros(2, c["Cout"], dtype=torch.float64, device=DEV)
    f = conv_fields(BF16, dict(c, res=False), g, o)
    f.update(res=buf.data_ptr(), ldr=c["Cout"])
    run(_lib.make_op(_lib.OP_CONV, **f))
    v = ref_conv_acc(g, c) + prior.double()
    assert_equal(buf, v, f"INPLACE_CASES[{i}] accumulated gradient")
    if bw:
        xhat = (g["bw_x"].double() - g["bw_mean"].double()) * g["bw_invstd"].double()
        check_bn_bwd_sums(o["stats"], v * (g["bw_act"].double() > 0), xhat, f"INPLACE_CASES[{i}]")
    pin = {p.replace("epi=0", "epi=2") for p in INPLACE_CASES[i]["pin"]} if bw else INPLACE_CASES[i]["pin"]
    assert_pinned(capfd, pin)


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(SLICED_CASES)))
def test_channel_sliced_dgrad_exact(verbose, capfd, i):
    """plan._dgrad_op with row0 / rows: the dgrad weights [cin][k*k*cout] offset by row0 rows, Cout = rows."""
    c = dict(SLICED_CASES[i], c1=0, up0=0)
    k, co, cin, row0, rows = c["k"], c["c0"], c["cin"], c["row0"], c["rows"]
    gen = torch.Generator().manual_seed(1000 + i)
    w_all = dev(_ints((cin, k * k * co), 2, gen), torch.bfloat16)
    dy = dev(_ints((c["B"], c["Hi"], c["Wi"], co), 2, gen), torch.bfloat16)
    out = torch.zeros(c["B"], c["Hi"], c["Wi"], rows, device=DEV, dtype=torch.bfloat16)
    cs = dict(c, Cout=rows)
    f = conv_fields(BF16, cs, {"src0": dy, "w": w_all}, {"out": out})
    f["w"] = w_all.data_ptr() + row0 * k * k * co * 2
    run(_lib.make_op(_lib.OP_CONV, **f))
    ref = ref_conv_acc({"src0": dy, "w": w_all[row0:row0 + rows]}, cs)
    assert_equal(out, ref, f"SLICED_CASES[{i}]")
    assert_pinned(capfd, c["pin"])


# ------------------------------------------------------------------ NCHW -> NHWC with the head-bias chansum
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("i", range(len(CHANSUM_CASES)))
def test_nchw2nhwc_chansum_exact(verbose, capfd, dtype, i):
    s = CHANSUM_CASES[i]
    B, H, W = s["B"], s["H"], s["W"]
    gen = torch.Generator().manual_seed(1100 + i)
    src = dev(_ints((B, 3, H, W), 2, gen))
    dst = torch.ones(B, H, W, 16, device=DEV, dtype=TDT[dtype])
    cs = torch.tensor([5.0, -3.0, 7.0], device=DEV)       # accumulates onto what the bias gradient already holds
    op = _lib.make_op(_lib.OP_NCHW2NHWC, dtype=dtype, B=B, C=3, H=H, W=W, cpad=16, src=src.data_ptr(), dst=dst.data_ptr(),
                      chansum=cs.data_ptr())
    run(op)
    ref = torch.zeros(B, H, W, 16, dtype=torch.float64, device=DEV)
    ref[..., :3] = src.double().permute(0, 2, 3, 1)
    assert_equal(dst, ref, "dst (pad channels zero)")
    assert 3 * B * H * W * 2 <= EXACT_LIMIT
    assert_equal(cs, src.double().sum((0, 2, 3)) + torch.tensor([5.0, -3.0, 7.0], device=DEV, dtype=torch.float64),
                 "chansum", "c")
    assert_pinned(capfd, set(op_classes(op)), op_classes(op))


# ------------------------------------------------------------------ BatchNorm backward with mask_from_x
def bn_bwd_inputs(dtype, C, count, seed):
    """Raw x (integers), published scale / shift / mean / invstd, and act = relu(fmaf(x, scale, shift)) from bn_apply."""
    gen = torch.Generator().manual_seed(seed)
    x = dev(_ints((count, C), 4, gen), TDT[dtype])
    gamma = dev(torch.rand(C, generator=gen) + 0.5)
    mean = dev(torch.randn(C, generator=gen) * 0.5)
    invstd = dev(torch.rand(C, generator=gen) + 0.5)
    beta = dev(torch.randn(C, generator=gen))
    scale = (gamma.double() * invstd.double()).float()
    shift = (beta.double() - mean.double() * scale.double()).float()
    act = torch.zeros_like(x)
    run(_lib.make_op(_lib.OP_BN_APPLY, dtype=dtype, C=C, relu=1, count=count, x=x.data_ptr(), ldx=C, y=act.data_ptr(), ldy=C,
                     scale=scale.data_ptr(), shift=shift.data_ptr()))
    mask = (x.double() * scale.double() + shift.double()) > 0
    assert torch.equal(act > 0, mask), "bn_apply's act > 0 differs from the float64 mask"
    dy = dev(_ints((count, C), 2, gen), TDT[dtype])
    return dict(x=x, act=act, dy=dy, gamma=gamma, mean=mean, invstd=invstd, scale=scale, shift=shift, mask=mask)


def bn_bwd_fields(dtype, C, count, d, mask_from_x, o):
    return dict(dtype=dtype, C=C, relu=1, mask_from_x=mask_from_x, count=count, x=d["x"].data_ptr(), ldx=C,
                gamma=d["gamma"].data_ptr(), mean=d["mean"].data_ptr(), invstd=d["invstd"].data_ptr(),
                scale=d["scale"].data_ptr(), shift=d["shift"].data_ptr(), dy=d["dy"].data_ptr(), lddy=C,
                act=d["act"].data_ptr(), ldact=C, dx=o["dx"].data_ptr(), lddx=C, dres=o["dres"].data_ptr(), lddres=C,
                bstats=o["bstats"].data_ptr(), dgamma=o["dgamma"].data_ptr(), dbeta=o["dbeta"].data_ptr(),
                coef=o["coef"].data_ptr())


def bn_bwd_outputs(dtype, C, count):
    z = lambda: torch.zeros(count, C, device=DEV, dtype=TDT[dtype])
    return dict(dx=z(), dres=z(), bstats=torch.zeros(2, C, dtype=torch.float64, device=DEV),
                dgamma=torch.zeros(C, device=DEV), dbeta=torch.zeros(C, device=DEV), coef=torch.zeros(3, C, device=DEV),
                barrier=torch.zeros(2, dtype=torch.int32, device=DEV))


def check_bn_bwd(d, o, gp, what, gp_sums=None):
    """dres = g' exactly; dgamma / dbeta = the sums (dbeta exact under the budget); dx per element within
    BF16_REL * |ref| + BN_BWD_FP32_OPS * U * |c0| * (|g'| + |c1| + |xhat * c2|), ref from the launch's own sums in float64."""
    n = gp.shape[0]
    assert_equal(o["dres"], gp, f"{what} dres (= masked dy)", "pc")
    xhat = (d["x"].double() - d["mean"].double()) * d["invstd"].double()
    check_bn_bwd_sums(o["bstats"], gp if gp_sums is None else gp_sums, xhat, what)
    assert_equal(o["dbeta"], o["bstats"][0].float(), f"{what} dbeta", "c")
    assert_equal(o["dgamma"], o["bstats"][1].float(), f"{what} dgamma", "c")
    c0 = d["gamma"].double() * d["invstd"].double()
    c1, c2 = o["bstats"][0] / n, o["bstats"][1] / n
    ref = c0 * (gp - c1 - xhat * c2)
    bound = BF16_REL * ref.abs() + BN_BWD_FP32_OPS * U * c0.abs() * (gp.abs() + c1.abs() + (xhat * c2).abs())
    assert_within(o["dx"], ref, bound, f"{what} dx", "pc")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C,count", BN_BWD_CASES)
@pytest.mark.parametrize("form", ["two_kernels", "barrier"])
@pytest.mark.parametrize("mask_from_x", [1, 0])
def test_bn_bwd_mask_from_x(verbose, capfd, dtype, C, count, form, mask_from_x):
    """D3FK_OP_BN_BWD (reduce + apply; `barrier` set as the plans set it) with the ReLU mask re-derived from x and the
    published scale / shift (mask_from_x = 1) or read from act (0): the mask equals the float64 mask and act > 0 exactly."""
    d = bn_bwd_inputs(dtype, C, count, 1200 + C + count)
    o = bn_bwd_outputs(dtype, C, count)
    f = bn_bwd_fields(dtype, C, count, d, mask_from_x, o)
    if form == "barrier":
        f["barrier"] = o["barrier"].data_ptr()
    op = _lib.make_op(_lib.OP_BN_BWD, **f)
    run(op)
    gp = d["dy"].double() * d["mask"]
    check_bn_bwd(d, o, gp, f"bn_bwd C={C} count={count}")
    assert_pinned(capfd, set(op_classes(op)), op_classes(op))


@pytest.mark.gpu
@pytest.mark.parametrize("i", [0, 4, 5])
def test_bn_bwd_apply_after_fused_dgrad(verbose, capfd, i):
    """plan._bn_bwd's `prod is not None` branch: a dgrad carrying the BN-backward sums (FUSE 2, mask from act) followed by
    D3FK_OP_BN_BWD_APPLY with mask_from_x — the two masks must agree, and dx follows from the dgrad's sums."""
    c = dict(BW_CASES[i], res=False, bw=None)
    C = c["Cout"]
    Ho, Wo = _out_hw(c)
    count = c["B"] * Ho * Wo
    d = bn_bwd_inputs(BF16, C, count, 1300 + i)
    t = exact_operands("conv", c, 1350 + i)
    g = {n: dev(v, torch.bfloat16) for n, v in t.items()}
    o = bn_bwd_outputs(BF16, C, count)
    grad = torch.zeros(c["B"], Ho, Wo, C, device=DEV, dtype=torch.bfloat16)
    f = conv_fields(BF16, c, g, {"out": grad})
    f.update(stats=o["bstats"].data_ptr(), bw_x=d["x"].data_ptr(), bw_act=d["act"].data_ptr(), bw_mean=d["mean"].data_ptr(),
             bw_invstd=d["invstd"].data_ptr(), bw_ldx=C, bw_ldact=C, bw_relu=1)
    run(_lib.make_op(_lib.OP_CONV, **f))
    v = ref_conv_acc(g, c)
    assert_equal(grad, v.reshape(c["B"], Ho, Wo, C), f"BW_CASES[{i}] dgrad")
    d["dy"] = grad.view(count, C)
    op = _lib.make_op(_lib.OP_BN_BWD_APPLY, **bn_bwd_fields(BF16, C, count, d, 1, o))
    run(op)
    # the dgrad's sums are over its fp32 value v (include/d3fk.h); the apply reads the stored bf16(v)
    check_bn_bwd(d, o, grad.view(count, C).double() * d["mask"], f"BW_CASES[{i}] + bn_bwd_apply",
                 gp_sums=v.reshape(count, C) * d["mask"])
    assert_pinned(capfd, PIN_BW[i] | set(op_classes(op)), op_classes(op))


# ------------------------------------------------------------------ coverage of the benchmarked plans
def declared_classes():
    out = set()
    for pins in (PIN_BW, PIN_GROUP, PIN_HEAD):
        for s in pins.values():
            out |= set(s)
    for table in (CONV_ALL, WGRAD_ALL, CONV_BN_ALL):
        for _, _, pin in table:
            out |= set(pin)
    for c in INPLACE_CASES:
        out |= set(c["pin"]) | {p.replace("epi=0", "epi=2") for p in c["pin"]}
    for c in SLICED_CASES + HALVES_CASES:
        out |= set(c["pin"])
    out |= STEM_PIN
    for dt in ("f32", "bf16"):
        out |= {f"nchw2nhwc<{dt}> chansum=1"}
        for xm in (0, 1):
            out |= {f"bn_bwd_reduce<{dt}> xmask={xm}", f"bn_bwd_apply<{dt}> xmask={xm}"}
    out |= {"head_conv<128>", "head_conv<64>", "head_conv<32>"}
    return out


PLANS = [("train", 256, 64), ("eval", 64, 128), ("train", 14, 128), ("train", 64, 128)]


@pytest.mark.gpu
def test_benchmarked_plans_only_launch_pinned_classes(verbose, capfd):
    """One step of each benchmarked plan (bf16 training at B = 256 @ 64^2, forward and backward through d3.Unet; the eval
    plan at B = 64 @ 128^2; the swap step's training plans at B = 14 and 64 @ 128^2) with the launch lines on: every class
    launched must be one an exact case above pins."""
    import denoising_diffusion_deep_fake_b200 as d3
    torch.manual_seed(0)
    m = d3.Unet(precision="bf16").to(DEV)
    seen = set()
    capfd.readouterr()
    for mode, B, H in PLANS:
        x = torch.randn(B, 3, H, H, device=DEV).clamp(-1, 1)
        if mode == "train":
            m.train()
            y = m(x)
            y.backward(torch.randn_like(y))
        else:
            m.eval()
            with torch.no_grad():
                m(x)
        torch.cuda.synchronize()
        seen |= set(launched_classes(capfd.readouterr().err))
    for plans in m._plans.values():
        for plan in plans:
            lists = [plan.pack_ops, plan.fwd_ops] + list(plan.bwd_segments or [])
            for ol in lists:
                for op in ol:
                    seen |= set(op_classes(op))
    print("PLAN CLASSES", sorted(seen))
    missing = seen - declared_classes()
    assert not missing, f"classes the benchmarked plans launch but no exact case pins: {sorted(missing)}"
