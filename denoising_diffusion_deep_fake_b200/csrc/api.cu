// api.cu — the extern "C" surface of libd3fk (declared in include/d3fk.h) and the op-list runner.
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>
#include "common.cuh"

namespace d3fk {

int64_t g_launch_count = 0;
char g_last_error[512] = "";
int* g_dev_error_flag = nullptr;
int g_use_pdl = 1;
static int g_inited_device = -1;

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
  va_end(ap);
  return code;
}

int check_launch(const char* what) {
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    cudaGetLastError();
    return set_error(D3FK_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  }
  return D3FK_OK;
}

// launchers implemented in the other translation units
int launch_conv_ffma(const d3fk_conv_params*, cudaStream_t);
int launch_wgrad_ffma(const d3fk_wgrad_params*, cudaStream_t);
int launch_conv_tc(const d3fk_conv_params*, cudaStream_t);
int launch_wgrad_tc(const d3fk_wgrad_params*, cudaStream_t);
int launch_wgrad_group_tc(const d3fk_wgrad_group_params*, cudaStream_t);
int launch_conv_bn_tc(const d3fk_convbn_params*, cudaStream_t);
int launch_pack(const d3fk_pack_params*, cudaStream_t);
int launch_nchw_to_nhwc(const d3fk_layout_params*, cudaStream_t);
int launch_nchw_to_s2d(const d3fk_layout_params*, cudaStream_t);
int launch_pack_stem(const d3fk_pack_params*, cudaStream_t);
int launch_bn_finalize(const d3fk_bn_params*, cudaStream_t);
int launch_bn_fold(const d3fk_bn_params*, cudaStream_t);
int launch_bn_apply(const d3fk_bn_params*, cudaStream_t);
int launch_bn_bwd_reduce(const d3fk_bn_params*, cudaStream_t);
int launch_bn_bwd_finalize(const d3fk_bn_params*, cudaStream_t);
int launch_bn_bwd_apply(const d3fk_bn_params*, cudaStream_t);
int launch_bn_bwd(const d3fk_bn_params*, cudaStream_t);
extern int g_fuse_bn_bwd;
extern long long g_fuse_bn_bwd_max;
int launch_maxpool_fwd(const d3fk_pool_params*, cudaStream_t);
int launch_maxpool_bwd(const d3fk_pool_params*, cudaStream_t);
int launch_sumpool2(const d3fk_pool_params*, cudaStream_t);
int launch_chansum(const d3fk_chansum_params*, cudaStream_t);
int launch_upcat(const d3fk_upcat_params*, cudaStream_t);
int launch_frames_to_tensor(const d3fk_frames_params*, cudaStream_t);
int launch_tensor_to_frames(const d3fk_frames_params*, cudaStream_t);
int launch_affine_qsample(const d3fk_affine_qsample_params*, cudaStream_t);
int launch_qsample(const d3fk_qsample_params*, cudaStream_t);
int launch_posterior(const d3fk_posterior_params*, cudaStream_t);
int launch_posterior_2m(const d3fk_posterior_2m_params*, cudaStream_t);
int launch_inc(const d3fk_misc_params*, cudaStream_t);
int launch_adam(const d3fk_adam_params*, cudaStream_t);
int launch_set_scalars(const d3fk_scalars_params*, cudaStream_t);
int launch_pack_all(const d3fk_misc_params*, cudaStream_t);
int launch_loss(const d3fk_loss_params*, cudaStream_t);
int loss_init();
int tc_init();

static int require_init() {
  if (g_inited_device < 0) return set_error(D3FK_ERR_ARCH, "d3fk_init() has not succeeded on an sm_100 device");
  return D3FK_OK;
}

static int conv_dispatch(const d3fk_conv_params* p, cudaStream_t s) {
  if (p->dtype == D3FK_F32) {
    if (p->mode == 2) return set_error(D3FK_ERR_UNSUPPORTED, "conv mode 2 (windowed rows) is a bf16-engine path");
    return launch_conv_ffma(p, s);
  }
  if (p->dtype == D3FK_BF16) return launch_conv_tc(p, s);
  return set_error(D3FK_ERR_ARG, "conv: bad dtype %d", p->dtype);
}
static int wgrad_dispatch(const d3fk_wgrad_params* p, cudaStream_t s) {
  if (p->dtype == D3FK_F32) {
    if (p->mode == 2) return set_error(D3FK_ERR_UNSUPPORTED, "wgrad mode 2 (space-to-depth stem) is a bf16-engine path");
    return launch_wgrad_ffma(p, s);
  }
  if (p->dtype == D3FK_BF16) return launch_wgrad_tc(p, s);
  return set_error(D3FK_ERR_ARG, "wgrad: bad dtype %d", p->dtype);
}

static int wgrad_group_dispatch(const d3fk_wgrad_group_params* p, cudaStream_t s) {
  if (p->base.dtype == D3FK_BF16) return launch_wgrad_group_tc(p, s);
  if (p->count < 1 || p->count > D3FK_WGRAD_GROUP_MAX) return set_error(D3FK_ERR_ARG, "wgrad group: count %d", p->count);
  for (int i = 0; i < p->count; ++i) {        // fp32 parity mode: one launch per problem
    d3fk_wgrad_params one = p->base;
    one.src0 = p->src0[i]; one.dy = p->dy[i]; one.dw = p->dw[i];
    int rc = wgrad_dispatch(&one, s);
    if (rc) return rc;
  }
  return D3FK_OK;
}

static int convbn_dispatch(const d3fk_convbn_params* p, cudaStream_t s) {
  if (p->conv.dtype == D3FK_BF16) return launch_conv_bn_tc(p, s);
  int rc = conv_dispatch(&p->conv, s);      // fp32 parity mode: the two kernels
  return rc ? rc : launch_bn_apply(&p->bn, s);
}

static int run_one(const d3fk_op* op, cudaStream_t s) {
  switch (op->kind) {
    case D3FK_OP_CONV_BN: return convbn_dispatch(&op->u.convbn, s);
    case D3FK_OP_CONV: return conv_dispatch(&op->u.conv, s);
    case D3FK_OP_WGRAD: return wgrad_dispatch(&op->u.wgrad, s);
    case D3FK_OP_WGRAD_GROUP: return wgrad_group_dispatch(&op->u.wgrad_group, s);
    case D3FK_OP_PACK: return launch_pack(&op->u.pack, s);
    case D3FK_OP_NCHW2NHWC: return launch_nchw_to_nhwc(&op->u.layout, s);
    case D3FK_OP_NCHW2S2D: return launch_nchw_to_s2d(&op->u.layout, s);
    case D3FK_OP_PACK_STEM: return launch_pack_stem(&op->u.pack, s);
    case D3FK_OP_BN_FINALIZE: return launch_bn_finalize(&op->u.bn, s);
    case D3FK_OP_BN_APPLY: return launch_bn_apply(&op->u.bn, s);
    case D3FK_OP_BN_FOLD: return launch_bn_fold(&op->u.bn, s);
    case D3FK_OP_BN_BWD_REDUCE: return launch_bn_bwd_reduce(&op->u.bn, s);
    case D3FK_OP_BN_BWD_FINALIZE: return launch_bn_bwd_finalize(&op->u.bn, s);
    case D3FK_OP_BN_BWD_APPLY: return launch_bn_bwd_apply(&op->u.bn, s);
    case D3FK_OP_BN_BWD: return launch_bn_bwd(&op->u.bn, s);
    case D3FK_OP_MAXPOOL_FWD: return launch_maxpool_fwd(&op->u.pool, s);
    case D3FK_OP_MAXPOOL_BWD: return launch_maxpool_bwd(&op->u.pool, s);
    case D3FK_OP_SUMPOOL2: return launch_sumpool2(&op->u.pool, s);
    case D3FK_OP_CHANSUM: return launch_chansum(&op->u.chansum, s);
    case D3FK_OP_UPCAT: return launch_upcat(&op->u.upcat, s);
    case D3FK_OP_FRAMES_TO_TENSOR: return launch_frames_to_tensor(&op->u.frames, s);
    case D3FK_OP_TENSOR_TO_FRAMES: return launch_tensor_to_frames(&op->u.frames, s);
    case D3FK_OP_AFFINE_QSAMPLE: return launch_affine_qsample(&op->u.affine_qsample, s);
    case D3FK_OP_QSAMPLE: return launch_qsample(&op->u.qsample, s);
    case D3FK_OP_POSTERIOR: return launch_posterior(&op->u.posterior, s);
    case D3FK_OP_POSTERIOR_2M: return launch_posterior_2m(&op->u.posterior_2m, s);
    case D3FK_OP_MEMSET: {
      cudaError_t e = cudaMemsetAsync(op->u.misc.p0, 0, (size_t)op->u.misc.n, s);
      if (e != cudaSuccess) return set_error(D3FK_ERR_CUDA, "memset: %s", cudaGetErrorString(e));
      return D3FK_OK;
    }
    case D3FK_OP_INC: return launch_inc(&op->u.misc, s);
    case D3FK_OP_ADAM: return launch_adam(&op->u.adam, s);
    case D3FK_OP_SET_SCALARS: return launch_set_scalars(&op->u.scalars, s);
    case D3FK_OP_JOIN: return D3FK_OK;      // stream bookkeeping of run_list; nothing to launch
    case D3FK_OP_PACK_ALL: return launch_pack_all(&op->u.misc, s);
    case D3FK_OP_LOSS: return launch_loss(&op->u.loss, s);
    default: return set_error(D3FK_ERR_ARG, "unknown op kind %d", op->kind);
  }
}

}  // namespace d3fk

using namespace d3fk;

extern "C" {

int d3fk_version(void) { return 2; }
int d3fk_sizeof_op(void) { return (int)sizeof(d3fk_op); }
const char* d3fk_last_error(void) { return g_last_error; }
int64_t d3fk_launch_count(void) { return g_launch_count; }

int d3fk_init(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    return set_error(D3FK_ERR_ARCH, "no CUDA device (%s); libd3fk has no CPU path", cudaGetErrorString(e));
  }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return set_error(D3FK_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
  if (prop.major != 10) return set_error(D3FK_ERR_ARCH, "device %d is sm_%d%d; libd3fk is sm_100a only", device, prop.major, prop.minor);
  if (!g_dev_error_flag) {
    const size_t dbg_bytes = 64 + 512 * 16 * sizeof(unsigned long long);   // error flag + (D3FK_TIMELINE builds) phase stamps
    e = cudaMalloc(&g_dev_error_flag, dbg_bytes);
    if (e != cudaSuccess) return set_error(D3FK_ERR_CUDA, "cudaMalloc: %s", cudaGetErrorString(e));
    cudaMemset(g_dev_error_flag, 0, dbg_bytes);
  }
  if (const char* v = getenv("D3FK_PDL")) g_use_pdl = atoi(v);     // launch attribute only: same kernels, same results
#ifdef D3FK_DEBUG
  if (const char* v = getenv("D3FK_FUSE_BN_BWD")) g_fuse_bn_bwd = atoi(v);
  if (const char* v = getenv("D3FK_FUSE_BN_BWD_MAX")) g_fuse_bn_bwd_max = atoll(v);
#endif
  int rc = tc_init();
  if (rc) return rc;
  rc = loss_init();
  if (rc) return rc;
  g_inited_device = device;
  return D3FK_OK;
}

/* debug: copy the first n 64-bit timeline words (D3FK_TIMELINE builds only write them) and the launch counter */
int d3fk_debug_timeline(unsigned long long* out, int n, unsigned* launches) {
  if (!g_dev_error_flag) return D3FK_ERR_ARG;
  cudaDeviceSynchronize();
  cudaMemcpy(out, g_dev_error_flag + 16, (size_t)n * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
  cudaMemcpy(launches, g_dev_error_flag + 4, sizeof(unsigned), cudaMemcpyDeviceToHost);
  return D3FK_OK;
}

int d3fk_device_error_flag(void) {
  if (!g_dev_error_flag) return 0;
  int v = 0;
  cudaMemcpy(&v, g_dev_error_flag, sizeof(int), cudaMemcpyDeviceToHost);
  return v;
}

// Weight gradients are off the backward critical path (dgrad_L -> BN-backward_{L-1} -> dgrad_{L-1} ...): d3fk_run forks
// every OP_WGRAD onto a side stream behind an event recorded after its producer and joins the side stream at the end of
// the op list, so the latency-bound deep-layer kernels of the two chains overlap.  Event record / wait are capture-safe.
constexpr int MAX_SIDE = 8;
static cudaStream_t g_side_streams[MAX_SIDE] = {nullptr};
static cudaEvent_t g_join_events[MAX_SIDE];
static int g_n_side = 1;       // D3FK_SIDE_STREAMS: ONE side stream — concurrent weight-gradient kernels only take more SM slots away from
                               // the main chain (measured: 3.84 ms/step with 3 streams, 3.77 with 1, 3.87 with 6)
static unsigned g_side_cursor = 0;
#define g_side_stream g_side_streams[0]
static cudaEvent_t g_fork_events[64];
static int g_n_fork_events = 0;
static unsigned g_fork_cursor = 0;
static bool g_side_pending = false;
#ifdef D3FK_DEBUG
static int g_skip_wgrad = 0;
#endif
static int g_fork_wgrad = 1;   // D3FK_FORK_WGRAD=0: everything in stream order
#define g_fork_lanes g_fork_wgrad

static cudaStream_t g_lane_streams[D3FK_MAX_LANES] = {nullptr};
static cudaEvent_t g_lane_events[D3FK_MAX_LANES];

static int ensure_side_stream() {
  if (g_side_stream) return D3FK_OK;
  if (const char* v = getenv("D3FK_FORK_WGRAD")) g_fork_wgrad = atoi(v);   // stream placement only
#ifdef D3FK_DEBUG
  if (const char* v = getenv("D3FK_SKIP_WGRAD")) g_skip_wgrad = atoi(v);   // timing experiment: DROPS work — debug builds only
#endif
  // (a higher-priority main stream was measured: no gain — both chains are latency-bound, not slot-bound)
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  if (const char* v = getenv("D3FK_SIDE_STREAMS")) g_n_side = atoi(v);
  if (g_n_side < 1) g_n_side = 1;
  if (g_n_side > MAX_SIDE) g_n_side = MAX_SIDE;
  cudaError_t e = cudaSuccess;
  for (int i = 0; i < g_n_side && e == cudaSuccess; ++i) {
    e = cudaStreamCreateWithPriority(&g_side_streams[i], cudaStreamNonBlocking, prio_lo);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g_join_events[i], cudaEventDisableTiming);
  }
  for (int i = 0; i < 64 && e == cudaSuccess; ++i) { e = cudaEventCreateWithFlags(&g_fork_events[i], cudaEventDisableTiming); g_n_fork_events = i + 1; }
  for (int i = 0; i < D3FK_MAX_LANES && e == cudaSuccess; ++i) {   // branch lanes: default priority, like the caller's stream
    e = cudaStreamCreateWithPriority(&g_lane_streams[i], cudaStreamNonBlocking, 0);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g_lane_events[i], cudaEventDisableTiming);
  }
  if (e != cudaSuccess) return set_error(D3FK_ERR_CUDA, "cudaEventCreate: %s", cudaGetErrorString(e));
  return D3FK_OK;
}


static int lane_join(int lane, cudaStream_t main, bool* open) {
  if (lane < 1 || lane > D3FK_MAX_LANES) return set_error(D3FK_ERR_ARG, "join: lane %d out of range", lane);
  if (!open[lane - 1]) return D3FK_OK;
  cudaError_t e = cudaEventRecord(g_lane_events[lane - 1], g_lane_streams[lane - 1]);
  if (e == cudaSuccess) e = cudaStreamWaitEvent(main, g_lane_events[lane - 1], 0);
  if (e != cudaSuccess) return set_error(D3FK_ERR_CUDA, "lane join: %s", cudaGetErrorString(e));
  open[lane - 1] = false;
  return D3FK_OK;
}

static int run_list(const d3fk_op* ops, int n_ops, cudaStream_t main_stream, bool join) {
  int rc = require_init();
  if (rc) return rc;
  rc = ensure_side_stream();
  if (rc) return rc;
  int forks = 0;
  bool lane_open[D3FK_MAX_LANES] = {false};
  for (int i = 0; i < n_ops; ++i) {
    if (ops[i].kind == D3FK_OP_JOIN) {
      rc = lane_join((int)ops[i].u.misc.n, main_stream, lane_open);
      if (rc) return rc;
      continue;
    }
    cudaStream_t s = main_stream;
    const int lane = ops[i].lane;
    if (lane != 0) {
      if (lane < 1 || lane > D3FK_MAX_LANES) return set_error(D3FK_ERR_ARG, "op %d: lane %d out of range", i, lane);
      if (!g_fork_lanes) {
        // D3FK_FORK_WGRAD=0 (everything in stream order) also keeps the branches on the main stream
      } else {
        s = g_lane_streams[lane - 1];
        if (!lane_open[lane - 1]) {            // fork: the branch starts behind what the main stream holds now
          cudaEvent_t ev = g_fork_events[g_fork_cursor++ % g_n_fork_events];
          cudaError_t e = cudaEventRecord(ev, main_stream);
          if (e == cudaSuccess) e = cudaStreamWaitEvent(s, ev, 0);
          if (e != cudaSuccess) return set_error(D3FK_ERR_CUDA, "lane fork: %s", cudaGetErrorString(e));
          lane_open[lane - 1] = true;
        }
      }
    }
    const bool is_wgrad = ops[i].kind == D3FK_OP_WGRAD || ops[i].kind == D3FK_OP_WGRAD_GROUP;
#ifdef D3FK_DEBUG
    if (is_wgrad && g_skip_wgrad) {           // timing experiment only (D3FK_SKIP_WGRAD: 1 = all; else 2 << class, class by pixel count)
      const d3fk_wgrad_params* wp = ops[i].kind == D3FK_OP_WGRAD ? &ops[i].u.wgrad : &ops[i].u.wgrad_group.base;
      const long long M = (long long)wp->B * wp->Ho * wp->Wo;
      const int cls = M >= 262144 ? 0 : M >= 65536 ? 1 : M >= 16384 ? 2 : M >= 4096 ? 3 : 4;
      if ((g_skip_wgrad & 1) || ((g_skip_wgrad >> (1 + cls)) & 1)) continue;
    }
#endif
    if (is_wgrad && g_fork_wgrad && n_ops > 1) {
      cudaEvent_t ev = g_fork_events[g_fork_cursor++ % g_n_fork_events];
      cudaStream_t side = g_side_streams[g_side_cursor++ % g_n_side];   // round robin: no false wgrad -> wgrad ordering
      cudaError_t e = cudaEventRecord(ev, s);
      if (e == cudaSuccess) e = cudaStreamWaitEvent(side, ev, 0);
      if (e != cudaSuccess) return set_error(D3FK_ERR_CUDA, "fork: %s", cudaGetErrorString(e));
      ++forks;
      rc = run_one(&ops[i], side);
    } else {
      rc = run_one(&ops[i], s);
    }
    if (rc) {
      char tmp[400];
      strncpy(tmp, g_last_error, sizeof(tmp) - 1);
      tmp[sizeof(tmp) - 1] = 0;
      return set_error(rc, "op %d (kind %d): %s", i, ops[i].kind, tmp);
    }
  }
  for (int l = 1; l <= D3FK_MAX_LANES; ++l) {      // a branch the list left open ends with the list
    rc = lane_join(l, main_stream, lane_open);
    if (rc) return rc;
  }
  if (forks) g_side_pending = true;
  if (join && g_side_pending) return d3fk_side_stream_join((d3fk_stream)main_stream);
  return D3FK_OK;
}

int d3fk_run(const d3fk_op* ops, int n_ops, d3fk_stream stream) { return run_list(ops, n_ops, (cudaStream_t)stream, true); }

/* as d3fk_run, but weight-gradient ops forked onto the side stream are NOT joined: the caller joins once, with
 * d3fk_side_stream_join, before anything consumes the weight gradients (optimizer step, gradient allreduce) */
int d3fk_run_nojoin(const d3fk_op* ops, int n_ops, d3fk_stream stream) { return run_list(ops, n_ops, (cudaStream_t)stream, false); }

int d3fk_side_stream_join(d3fk_stream stream) {
  if (!g_side_streams[0]) return D3FK_OK;
  for (int i = 0; i < g_n_side; ++i) {
    cudaError_t e = cudaEventRecord(g_join_events[i], g_side_streams[i]);
    if (e == cudaSuccess) e = cudaStreamWaitEvent((cudaStream_t)stream, g_join_events[i], 0);
    if (e != cudaSuccess) return set_error(D3FK_ERR_CUDA, "join: %s", cudaGetErrorString(e));
  }
  g_side_pending = false;
  return D3FK_OK;
}

// profiling aid: per-op device time with CUDA events (allocates events; not for the hot path)
int d3fk_run_profile(const d3fk_op* ops, int n_ops, d3fk_stream stream, float* ms_per_op) {
  int rc = require_init();
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  cudaEvent_t* ev = new cudaEvent_t[n_ops + 1];
  for (int i = 0; i <= n_ops; ++i) cudaEventCreate(&ev[i]);
  for (int i = 0; i < n_ops; ++i) {
    cudaEventRecord(ev[i], s);
    rc = run_one(&ops[i], s);
    if (rc) break;
  }
  cudaEventRecord(ev[n_ops], s);
  cudaStreamSynchronize(s);
  if (!rc)
    for (int i = 0; i < n_ops; ++i) cudaEventElapsedTime(&ms_per_op[i], ev[i], ev[i + 1]);
  for (int i = 0; i <= n_ops; ++i) cudaEventDestroy(ev[i]);
  delete[] ev;
  return rc;
}

#define SINGLE(name, type, fn)                                   \
  int name(const type* p, d3fk_stream stream) {                  \
    int rc = require_init();                                     \
    if (rc) return rc;                                           \
    return fn(p, (cudaStream_t)stream);                          \
  }
SINGLE(d3fk_conv, d3fk_conv_params, conv_dispatch)
SINGLE(d3fk_wgrad, d3fk_wgrad_params, wgrad_dispatch)
SINGLE(d3fk_wgrad_group, d3fk_wgrad_group_params, wgrad_group_dispatch)
SINGLE(d3fk_conv_bn, d3fk_convbn_params, convbn_dispatch)
SINGLE(d3fk_pack_weights, d3fk_pack_params, launch_pack)
SINGLE(d3fk_nchw_to_nhwc, d3fk_layout_params, launch_nchw_to_nhwc)
SINGLE(d3fk_bn_finalize, d3fk_bn_params, launch_bn_finalize)
SINGLE(d3fk_bn_apply, d3fk_bn_params, launch_bn_apply)
SINGLE(d3fk_bn_fold, d3fk_bn_params, launch_bn_fold)
SINGLE(d3fk_bn_bwd_reduce, d3fk_bn_params, launch_bn_bwd_reduce)
SINGLE(d3fk_bn_bwd_finalize, d3fk_bn_params, launch_bn_bwd_finalize)
SINGLE(d3fk_bn_bwd_apply, d3fk_bn_params, launch_bn_bwd_apply)
SINGLE(d3fk_bn_bwd, d3fk_bn_params, launch_bn_bwd)
SINGLE(d3fk_maxpool_fwd, d3fk_pool_params, launch_maxpool_fwd)
SINGLE(d3fk_maxpool_bwd, d3fk_pool_params, launch_maxpool_bwd)
SINGLE(d3fk_sumpool2, d3fk_pool_params, launch_sumpool2)
SINGLE(d3fk_chansum, d3fk_chansum_params, launch_chansum)
SINGLE(d3fk_upcat, d3fk_upcat_params, launch_upcat)
SINGLE(d3fk_frames_to_tensor, d3fk_frames_params, launch_frames_to_tensor)
SINGLE(d3fk_tensor_to_frames, d3fk_frames_params, launch_tensor_to_frames)
SINGLE(d3fk_affine_q_sample, d3fk_affine_qsample_params, launch_affine_qsample)
SINGLE(d3fk_q_sample, d3fk_qsample_params, launch_qsample)
SINGLE(d3fk_posterior_step, d3fk_posterior_params, launch_posterior)
SINGLE(d3fk_posterior_2m_step, d3fk_posterior_2m_params, launch_posterior_2m)
SINGLE(d3fk_adam, d3fk_adam_params, launch_adam)
SINGLE(d3fk_set_scalars, d3fk_scalars_params, launch_set_scalars)
SINGLE(d3fk_mse_ssim_loss, d3fk_loss_params, launch_loss)

}  // extern "C"
