"""ctypes binding of libd3fk.so (include/d3fk.h).  There is no fallback: if the shared library is
missing, or the device is not sm_100, every product entry point raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("D3FK_LIB", os.path.join(_HERE, "libd3fk.so"))   # D3FK_LIB: instrumented debug builds (tools/)

F32, BF16 = 0, 1

i32, i64, u64, f32, vp = C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_void_p


class ConvParams(C.Structure):
    _fields_ = [("dtype", i32), ("mode", i32), ("src0", vp), ("src1", vp),
                ("c0", i32), ("c1", i32), ("ld0", i32), ("ld1", i32), ("up0", i32),
                ("B", i32), ("Hi", i32), ("Wi", i32), ("Ho", i32), ("Wo", i32),
                ("kh", i32), ("kw", i32), ("stride", i32), ("pad", i32),
                ("w", vp), ("Cout", i32), ("_pad0", i32),
                ("out", vp), ("out_nchw", vp), ("scale", vp), ("shift", vp), ("res", vp), ("stats", vp),
                ("ldo", i32), ("ldr", i32), ("relu", i32), ("_pad1", i32), ("ws", vp), ("ws_bytes", i64),
                ("bw_x", vp), ("bw_act", vp), ("bw_mean", vp), ("bw_invstd", vp),
                ("bw_ldx", i32), ("bw_ldact", i32), ("bw_relu", i32), ("_pad2", i32)]


class WgradParams(C.Structure):
    _fields_ = [("dtype", i32), ("mode", i32), ("src0", vp), ("src1", vp),
                ("c0", i32), ("c1", i32), ("ld0", i32), ("ld1", i32), ("up0", i32),
                ("B", i32), ("Hi", i32), ("Wi", i32), ("Ho", i32), ("Wo", i32),
                ("kh", i32), ("kw", i32), ("stride", i32), ("pad", i32),
                ("dy", vp), ("dw", vp), ("ldy", i32), ("Cout", i32), ("cin_real", i32), ("cout_real", i32)]


WGRAD_GROUP_MAX = 12


class WgradGroupParams(C.Structure):
    _fields_ = [("base", WgradParams), ("count", i32), ("_pad0", i32),
                ("src0", vp * WGRAD_GROUP_MAX), ("dy", vp * WGRAD_GROUP_MAX), ("dw", vp * WGRAD_GROUP_MAX)]


class FramesParams(C.Structure):
    _fields_ = [("N", i32), ("H", i32), ("W", i32), ("_pad0", i32), ("frames", vp), ("tensor", vp),
                ("mean", C.c_float * 3), ("std", C.c_float * 3)]


class AffineQsampleParams(C.Structure):
    _fields_ = [("B", i32), ("C", i32), ("H", i32), ("W", i32), ("lam", f32), ("fixed_r", f32),
                ("x", vp), ("minv", vp), ("noise", vp), ("y", vp), ("out_aug", vp), ("out_noisy", vp), ("r_out", vp),
                ("seed", u64), ("offset", u64)]


class PackParams(C.Structure):
    _fields_ = [("dtype", i32), ("Cout", i32), ("Cin", i32), ("kh", i32), ("kw", i32), ("cin_pad", i32),
                ("cout_pad", i32), ("blk0", i32), ("w", vp), ("w_fwd", vp), ("w_dgrad", vp)]


class BnParams(C.Structure):
    _fields_ = [("dtype", i32), ("C", i32), ("relu", i32), ("mask_from_x", i32), ("count", i64),
                ("x", vp), ("y", vp), ("res", vp),
                ("ldx", i32), ("ldy", i32), ("ldr", i32), ("frozen", i32),
                ("stats", vp), ("gamma", vp), ("beta", vp),
                ("running_mean", vp), ("running_var", vp), ("num_batches_tracked", vp),
                ("eps", f32), ("momentum", f32),
                ("scale", vp), ("shift", vp), ("mean", vp), ("invstd", vp),
                ("dy", vp), ("act", vp), ("dx", vp), ("dres", vp),
                ("lddy", i32), ("ldact", i32), ("lddx", i32), ("lddres", i32),
                ("bstats", vp), ("dgamma", vp), ("dbeta", vp), ("coef", vp), ("barrier", vp)]


class PoolParams(C.Structure):
    _fields_ = [("dtype", i32), ("B", i32), ("H", i32), ("W", i32), ("C", i32), ("accumulate", i32),
                ("x", vp), ("y", vp), ("idx", vp), ("dy", vp), ("dx", vp),
                ("ldx", i32), ("ldy", i32), ("lddy", i32), ("lddx", i32)]


class LayoutParams(C.Structure):
    _fields_ = [("dtype", i32), ("B", i32), ("C", i32), ("H", i32), ("W", i32), ("cpad", i32), ("src", vp), ("dst", vp),
                ("chansum", vp)]


class ChansumParams(C.Structure):
    _fields_ = [("dtype", i32), ("C", i32), ("ld", i32), ("_pad0", i32), ("count", i64), ("x", vp), ("out", vp)]


class QsampleParams(C.Structure):
    _fields_ = [("B", i32), ("chw", i32), ("lam", f32), ("fixed_r", f32), ("x", vp), ("noise", vp), ("y", vp),
                ("out", vp), ("r_out", vp), ("noise_out", vp), ("seed", u64), ("offset", u64)]


class PosteriorParams(C.Structure):
    _fields_ = [("n", i64), ("x", vp), ("x0_hat", vp), ("z", vp), ("coef_table", vp), ("step", vp),
                ("k_xi", f32), ("k_x0", f32), ("sigma", f32), ("_pad0", f32), ("seed", u64), ("offset", u64)]


class MiscParams(C.Structure):
    _fields_ = [("p0", vp), ("n", i64)]


class AdamParams(C.Structure):
    _fields_ = [("n", i64), ("p", vp), ("g", vp), ("m", vp), ("v", vp), ("ema", vp),
                ("lr", f32), ("beta1", f32), ("beta2", f32), ("eps", f32), ("bias1", f32), ("bias2", f32),
                ("ema_decay", f32), ("grad_scale", f32), ("dyn", vp)]


class ScalarsParams(C.Structure):
    _fields_ = [("dst", vp), ("v", f32 * 4)]


class LossParams(C.Structure):
    _fields_ = [("B", i32), ("C", i32), ("H", i32), ("W", i32), ("pred", vp), ("target", vp), ("grad", vp), ("acc", vp),
                ("lo", f32), ("hi", f32), ("grad_scale", f32), ("_pad0", f32), ("win", f32 * 12), ("loss_out", vp)]


class ConvBnParams(C.Structure):
    _fields_ = [("conv", ConvParams), ("bn", BnParams), ("barrier", vp)]


class UpcatParams(C.Structure):
    _fields_ = [("dtype", i32), ("B", i32), ("H", i32), ("W", i32), ("c0", i32), ("c1", i32), ("ld0", i32), ("ld1", i32),
                ("ldo", i32), ("_pad0", i32), ("src0", vp), ("src1", vp), ("out", vp)]


class _OpUnion(C.Union):
    _fields_ = [("conv", ConvParams), ("wgrad", WgradParams), ("pack", PackParams), ("bn", BnParams),
                ("pool", PoolParams), ("layout", LayoutParams), ("chansum", ChansumParams),
                ("qsample", QsampleParams), ("posterior", PosteriorParams), ("misc", MiscParams),
                ("adam", AdamParams), ("loss", LossParams), ("convbn", ConvBnParams), ("upcat", UpcatParams),
                ("wgrad_group", WgradGroupParams), ("frames", FramesParams),
                ("affine_qsample", AffineQsampleParams), ("scalars", ScalarsParams)]


class Op(C.Structure):
    _fields_ = [("kind", i32), ("lane", i32), ("u", _OpUnion)]


# op kinds (enum d3fk_op_kind)
(OP_CONV, OP_WGRAD, OP_PACK, OP_NCHW2NHWC, OP_BN_FINALIZE, OP_BN_APPLY, OP_BN_FOLD, OP_BN_BWD_REDUCE,
 OP_BN_BWD_FINALIZE, OP_BN_BWD_APPLY, OP_MAXPOOL_FWD, OP_MAXPOOL_BWD, OP_SUMPOOL2, OP_CHANSUM, OP_QSAMPLE,
 OP_POSTERIOR, OP_MEMSET, OP_INC, OP_ADAM, OP_PACK_ALL, OP_LOSS, OP_CONV_BN, OP_UPCAT, OP_BN_BWD, OP_WGRAD_GROUP, OP_FRAMES_TO_TENSOR, OP_TENSOR_TO_FRAMES,
 OP_AFFINE_QSAMPLE, OP_SET_SCALARS, OP_JOIN) = range(1, 31)
OP_NCHW2S2D, OP_PACK_STEM = 31, 32
MAX_LANES = 2

_UNION_FIELD = {OP_CONV: "conv", OP_WGRAD: "wgrad", OP_PACK: "pack", OP_NCHW2NHWC: "layout",
                OP_BN_FINALIZE: "bn", OP_BN_APPLY: "bn", OP_BN_FOLD: "bn", OP_BN_BWD_REDUCE: "bn",
                OP_BN_BWD_FINALIZE: "bn", OP_BN_BWD_APPLY: "bn", OP_MAXPOOL_FWD: "pool", OP_MAXPOOL_BWD: "pool",
                OP_SUMPOOL2: "pool", OP_CHANSUM: "chansum", OP_QSAMPLE: "qsample", OP_POSTERIOR: "posterior",
                OP_MEMSET: "misc", OP_INC: "misc", OP_ADAM: "adam", OP_PACK_ALL: "misc",
                OP_LOSS: "loss", OP_CONV_BN: "convbn", OP_UPCAT: "upcat", OP_BN_BWD: "bn",
                OP_WGRAD_GROUP: "wgrad_group", OP_FRAMES_TO_TENSOR: "frames", OP_TENSOR_TO_FRAMES: "frames",
                OP_AFFINE_QSAMPLE: "affine_qsample", OP_SET_SCALARS: "scalars", OP_JOIN: "misc",
                OP_NCHW2S2D: "layout", OP_PACK_STEM: "pack"}
_PARAM_CLS = {"conv": ConvParams, "wgrad": WgradParams, "pack": PackParams, "bn": BnParams, "pool": PoolParams,
              "layout": LayoutParams, "chansum": ChansumParams, "qsample": QsampleParams,
              "posterior": PosteriorParams, "misc": MiscParams, "adam": AdamParams, "loss": LossParams,
              "convbn": ConvBnParams, "upcat": UpcatParams, "wgrad_group": WgradGroupParams,
              "frames": FramesParams, "affine_qsample": AffineQsampleParams, "scalars": ScalarsParams}

SINGLE_ENTRY = {OP_CONV: "d3fk_conv", OP_WGRAD: "d3fk_wgrad", OP_PACK: "d3fk_pack_weights",
                OP_NCHW2NHWC: "d3fk_nchw_to_nhwc", OP_BN_FINALIZE: "d3fk_bn_finalize", OP_BN_APPLY: "d3fk_bn_apply",
                OP_BN_FOLD: "d3fk_bn_fold", OP_BN_BWD_REDUCE: "d3fk_bn_bwd_reduce",
                OP_BN_BWD_FINALIZE: "d3fk_bn_bwd_finalize", OP_BN_BWD_APPLY: "d3fk_bn_bwd_apply",
                OP_MAXPOOL_FWD: "d3fk_maxpool_fwd", OP_MAXPOOL_BWD: "d3fk_maxpool_bwd", OP_SUMPOOL2: "d3fk_sumpool2",
                OP_CHANSUM: "d3fk_chansum", OP_QSAMPLE: "d3fk_q_sample", OP_POSTERIOR: "d3fk_posterior_step",
                OP_ADAM: "d3fk_adam", OP_LOSS: "d3fk_mse_ssim_loss", OP_CONV_BN: "d3fk_conv_bn", OP_UPCAT: "d3fk_upcat", OP_BN_BWD: "d3fk_bn_bwd",
                OP_WGRAD_GROUP: "d3fk_wgrad_group", OP_FRAMES_TO_TENSOR: "d3fk_frames_to_tensor",
                OP_TENSOR_TO_FRAMES: "d3fk_tensor_to_frames", OP_AFFINE_QSAMPLE: "d3fk_affine_q_sample",
                OP_SET_SCALARS: "d3fk_set_scalars"}
EXPORTS = ["d3fk_version", "d3fk_sizeof_op", "d3fk_init", "d3fk_last_error", "d3fk_device_error_flag", "d3fk_run",
           "d3fk_run_nojoin", "d3fk_side_stream_join", "d3fk_run_profile", "d3fk_launch_count", "d3fk_debug_timeline"] + sorted(set(SINGLE_ENTRY.values()))


def _set_fields(struct, fields):
    valid = {f[0] for f in struct._fields_}
    for k, v in fields.items():
        if k not in valid:
            raise KeyError(f"{type(struct).__name__} has no field {k!r}")
        if isinstance(v, dict):
            _set_fields(getattr(struct, k), v)      # nested POD (d3fk_convbn_params.conv / .bn)
        elif isinstance(v, (list, tuple)):          # pointer arrays (d3fk_wgrad_group_params)
            arr = getattr(struct, k)
            for i, x in enumerate(v):
                arr[i] = x
        else:
            setattr(struct, k, v)


def make_op(kind, lane=0, **fields):
    """Build one d3fk_op record.  Pointer fields take ints (tensor.data_ptr()) or None; nested structs take dicts.
    lane: 0 = the caller's stream, 1..MAX_LANES = a branch stream of d3fk_run (d3fk_op.lane)."""
    op = Op()
    op.kind = kind
    op.lane = lane
    _set_fields(getattr(op.u, _UNION_FIELD[kind]), fields)
    return op


def op_params(op):
    return getattr(op.u, _UNION_FIELD[op.kind])


class D3fkError(RuntimeError):
    pass


_lib = None
_inited = set()


def load():
    """Load libd3fk.so (no device needed).  Raises if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise D3fkError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        f"(there is no CPU or PyTorch fallback for the d3fk hot path)")
    lib = C.CDLL(LIB_PATH)
    lib.d3fk_last_error.restype = C.c_char_p
    lib.d3fk_launch_count.restype = C.c_int64
    lib.d3fk_run.argtypes = [C.POINTER(Op), C.c_int, vp]
    lib.d3fk_run_nojoin.argtypes = [C.POINTER(Op), C.c_int, vp]
    lib.d3fk_side_stream_join.argtypes = [vp]
    lib.d3fk_init.argtypes = [C.c_int]
    lib.d3fk_run_profile.argtypes = [C.POINTER(Op), C.c_int, vp, C.POINTER(C.c_float)]
    for kind, name in SINGLE_ENTRY.items():
        getattr(lib, name).argtypes = [C.POINTER(_PARAM_CLS[_UNION_FIELD[kind]]), vp]
    if lib.d3fk_sizeof_op() != C.sizeof(Op):
        raise D3fkError(f"ABI mismatch: sizeof(d3fk_op) = {lib.d3fk_sizeof_op()} in the library, "
                        f"{C.sizeof(Op)} in the Python mirror")
    _lib = lib
    return lib


def init(device_index):
    lib = load()
    if device_index in _inited:
        return lib
    rc = lib.d3fk_init(int(device_index))
    if rc != 0:
        raise D3fkError(f"d3fk_init({device_index}) failed ({rc}): {lib.d3fk_last_error().decode()}")
    _inited.add(device_index)
    return lib


def check(rc):
    if rc != 0:
        raise D3fkError(f"libd3fk error {rc}: {_lib.d3fk_last_error().decode()}")


class OpList:
    """A recorded op list: a contiguous ctypes array handed to d3fk_run in one call."""

    def __init__(self, ops):
        self.n = len(ops)
        self.array = (Op * max(self.n, 1))(*ops)

    def run(self, stream_ptr, join=True):
        """join=False: weight-gradient ops stay on libd3fk's side stream; call side_stream_join() before reading them."""
        if join:
            check(_lib.d3fk_run(self.array, self.n, stream_ptr))
        else:
            check(_lib.d3fk_run_nojoin(self.array, self.n, stream_ptr))

    def profile(self, stream_ptr):
        """Per-op device milliseconds (CUDA events around every op; synchronises)."""
        ms = (C.c_float * max(self.n, 1))()
        check(_lib.d3fk_run_profile(self.array, self.n, stream_ptr, ms))
        return list(ms)[:self.n]

    def __len__(self):
        return self.n

    def __iter__(self):
        return (self.array[i] for i in range(self.n))


def side_stream_join(stream_ptr):
    """Make `stream_ptr` wait for every weight-gradient kernel forked so far."""
    check(load().d3fk_side_stream_join(stream_ptr))


def run_single(op, stream_ptr):
    """Run one op through its dedicated extern "C" entry point (per-op parity tests)."""
    if op.kind in SINGLE_ENTRY:
        fn = getattr(_lib, SINGLE_ENTRY[op.kind])
        check(fn(C.byref(op_params(op)), stream_ptr))
    else:
        arr = (Op * 1)(op)
        check(_lib.d3fk_run(arr, 1, stream_ptr))


def launch_count():
    return int(load().d3fk_launch_count())
