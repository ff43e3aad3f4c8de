// elementwise.cu — bandwidth-bound passes of the d3f U-Net hot path (sm_100a).
//   BatchNorm(+residual)+ReLU apply / backward, statistics finalisation, max-pool, 2x2 sum-pool,
//   layout conversion, q_sample, posterior update, fused Adam(+EMA).
// All tensors are NHWC with 16-byte vector access (C is a multiple of 8); grids are sized in
// multiples of the SM count and loop grid-stride.
#include "common.cuh"

namespace d3fk {

static constexpr int kSMs = 148;
int g_fuse_bn_bwd = 0;   // D3FK_FUSE_BN_BWD=1: BN backward as one kernel behind a grid barrier (measured: no faster than two PDL launches)
long long g_fuse_bn_bwd_max = 4ll << 20;   // D3FK_FUSE_BN_BWD_MAX: largest tensor (elements) that takes the one-launch form
static inline int grid_for(long long work_items, int threads, int max_waves = 8) {
  long long blocks = (work_items + threads - 1) / threads;
  long long cap = (long long)kSMs * max_waves;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

// Occupancy of the BatchNorm kernels (bf16 engine): at the 110-126 registers ptxas picks on its own only two blocks fit
// an SM and the backward kernels reached 33-37 % of the HBM peak (ncu, r01e); capping the registers buys the third / fourth block.
#ifndef D3FK_BN_BWD_BLOCKS
#define D3FK_BN_BWD_BLOCKS 3
#endif
#define BN_BWD_OCC(T) (sizeof(T) == 2 ? D3FK_BN_BWD_BLOCKS : 1)

// ---------------------------------------------------------------------------------------------
// NCHW fp32 -> NHWC T, channels zero-padded to cpad (a multiple of 8)
// chansum (nullable, C <= 8): per-channel sums of the rounded values written, accumulated with one atomic per warp and channel
// (the head's bias gradient: saves the separate pass over dst).
template <typename T>
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ src, T* __restrict__ dst, int B, int C, int HW, int cpad, float* chansum) {
  pdl_enter();
  long long total = (long long)B * HW;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < total; p += (long long)gridDim.x * blockDim.x) {
    long long n = p / HW;
    long long hw = p - n * HW;
    const float* s = src + (n * C) * HW + hw;
    T* d = dst + p * cpad;
    constexpr int V = Vec<T>::N;
    for (int c0 = 0; c0 < cpad; c0 += V) {
      float v[V];
#pragma unroll
      for (int i = 0; i < V; ++i) v[i] = (c0 + i < C) ? __ldg(s + (long long)(c0 + i) * HW) : 0.f;
      store_vec<T>(d + c0, v);
      if (chansum && c0 < 8) {
#pragma unroll
        for (int i = 0; i < V; ++i)
          if (c0 + i < 8) acc[c0 + i] += to_f<T>(from_f<T>(v[i]));
      }
    }
  }
  if (chansum) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float a = acc[i];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
      if ((threadIdx.x & 31) == 0 && i < C) atomicAdd(chansum + i, a);
    }
  }
}

// fp32 NCHW (3 channels) -> the padded space-to-depth image the stem convolution (conv mode 2) reads: one thread per
// space-to-depth pixel (2x2 image pixels x 4 channels = 32 bytes).  Pad pixels and the 4th channel stay as allocated (zero).
__global__ void __launch_bounds__(256) nchw_to_s2d_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int B, int H, int W) {
  pdl_enter();
  const int Hs = H >> 1, Ws = W >> 1;
  const long long total = (long long)B * Hs * Ws;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int ws = (int)(i % Ws);
    const long long t = i / Ws;
    const int hs = (int)(t % Hs), b = (int)(t / Hs);
    float v[16];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float* p = src + (((long long)b * 3 + c) * H + 2 * hs) * W + 2 * ws;
      const float2 r0 = *reinterpret_cast<const float2*>(p), r1 = *reinterpret_cast<const float2*>(p + W);
      v[0 * 4 + c] = r0.x; v[1 * 4 + c] = r0.y; v[2 * 4 + c] = r1.x; v[3 * 4 + c] = r1.y;
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q * 4 + 3] = 0.f;
    __nv_bfloat16* d = dst + (((long long)b * Hs + hs) * (Ws + 3) + ws + 2) * 16;
    store_vec<__nv_bfloat16>(d, v);
    store_vec<__nv_bfloat16>(d + 8, v + 8);
  }
}
// 7x7 / stride-2 stem weights -> the [Cout][4 (th)][4 (tw)][2x2 (dy, dx)][4 (ci)] operand of conv mode 2
__global__ void pack_stem_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int Cout) {
  pdl_enter();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Cout * 256) return;
  const int co = i >> 8, k = i & 255;
  const int th = k >> 6, tw = (k >> 4) & 3, dy = (k >> 3) & 1, dx = (k >> 2) & 1, ci = k & 3;
  const int kh = 2 * th + dy - 1, kw = 2 * tw + dx - 1;
  float v = 0.f;
  if (ci < 3 && kh >= 0 && kh < 7 && kw >= 0 && kw < 7) v = w[((co * 3 + ci) * 7 + kh) * 7 + kw];
  out[i] = __float2bfloat16_rn(v);
}

// ---------------------------------------------------------------------------------------------
// BN statistics -> scale/shift, saved mean/invstd, running-stat update (momentum, unbiased var)
__global__ void bn_finalize_kernel(d3fk_bn_params p) {
  pdl_enter();
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= p.C) return;
  double n = (double)p.count;
  double mean = p.stats[c] / n;
  double var = p.stats[p.C + c] / n - mean * mean;
  if (var < 0) var = 0;
  double invstd = 1.0 / sqrt(var + (double)p.eps);
  float g = p.gamma[c], b = p.beta[c];
  float sc = (float)((double)g * invstd);
  p.scale[c] = sc;
  p.shift[c] = (float)((double)b - mean * (double)g * invstd);
  p.mean[c] = (float)mean;
  p.invstd[c] = (float)invstd;
  if (p.running_mean) {
    double unbiased = n > 1 ? var * n / (n - 1) : var;
    p.running_mean[c] = (float)((1.0 - p.momentum) * p.running_mean[c] + p.momentum * mean);
    p.running_var[c] = (float)((1.0 - p.momentum) * p.running_var[c] + p.momentum * unbiased);
  }
  if (c == 0 && p.num_batches_tracked) *p.num_batches_tracked += 1;
}

// eval mode: scale/shift from running statistics (folded into the conv epilogue).  mean / invstd set (frozen-BN plans): the
// running statistics are published there too, for the backward's xhat = (x - running_mean) * invstd_run.
__global__ void bn_fold_kernel(d3fk_bn_params p) {
  pdl_enter();
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= p.C) return;
  float invstd = 1.0f / sqrtf(p.running_var[c] + p.eps);
  float sc = p.gamma[c] * invstd;
  p.scale[c] = sc;
  p.shift[c] = p.beta[c] - p.running_mean[c] * sc;
  if (p.mean) p.mean[c] = p.running_mean[c];
  if (p.invstd) p.invstd[c] = invstd;
}

// y = relu?(x*scale + shift + res).  With p.stats set (train forward) the batch statistics are finalised here:
// every thread derives scale/shift of its own 8 (4) channels from the conv-epilogue sums, and the first C/V
// threads of block 0 publish mean / invstd / running statistics — no separate finalize launch.
template <typename T>
__global__ void __launch_bounds__(256, BN_BWD_OCC(T)) bn_apply_kernel(d3fk_bn_params p) {
  pdl_enter();
  constexpr int V = Vec<T>::N;
  constexpr int U = 4;               // independent 16-byte loads in flight per thread
  const int cvs = p.C / V;
  const long long total = p.count * cvs;
  const T* x = (const T*)p.x;
  T* y = (T*)p.y;
  const T* res = (const T*)p.res;
  const long long e0 = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;   // multiple of cvs: the channel vector is loop invariant
  const int c = (int)(e0 % cvs) * V;
  uint4 vr[U], rr[U];                // held packed (4 registers per vector) until used: 3 blocks per SM instead of 2
  // the pixel of element e0 + k * stride is pix0 + k * pstep (stride is a multiple of cvs): no division per vector
  const long long pix0 = e0 / cvs, pstep = stride / cvs;
  auto load_batch = [&](long long e, long long pixb) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long eu = e + u * stride;
      if (eu < total) {
        const long long pix = pixb + u * pstep;
        vr[u] = load_raw<T>(x + pix * p.ldx + c);
        if (res) rr[u] = load_raw<T>(res + pix * p.ldr + c);
      }
    }
  };
  load_batch(e0, pix0);              // first loads are in flight while the block derives scale / shift
  extern __shared__ float s_aff[];   // [2][C] scale, shift — derived once per block
  for (int ch = threadIdx.x; ch < p.C; ch += blockDim.x) {
    float sc, sh;
    if (p.stats) {
      const double n = (double)p.count;
      const double mean = p.stats[ch] / n;
      double var = p.stats[p.C + ch] / n - mean * mean;
      if (var < 0) var = 0;
      const double invstd = rsqrt(var + (double)p.eps);
      const double g = (double)p.gamma[ch], b = (double)p.beta[ch];
      sc = (float)(g * invstd);
      sh = (float)(b - mean * g * invstd);
      if (blockIdx.x == 0) {
        p.mean[ch] = (float)mean;
        p.invstd[ch] = (float)invstd;
        if (p.scale) { p.scale[ch] = sc; p.shift[ch] = sh; }   // backward re-derives the ReLU mask from them (mask_from_x)
        if (p.running_mean) {
          const double unbiased = n > 1 ? var * n / (n - 1) : var;
          p.running_mean[ch] = (float)((1.0 - p.momentum) * p.running_mean[ch] + p.momentum * mean);
          p.running_var[ch] = (float)((1.0 - p.momentum) * p.running_var[ch] + p.momentum * unbiased);
        }
        if (ch == 0 && p.num_batches_tracked) *p.num_batches_tracked += 1;
      }
    } else {
      sc = __ldg(p.scale + ch);
      sh = __ldg(p.shift + ch);
    }
    s_aff[ch] = sc;
    s_aff[p.C + ch] = sh;
  }
  __syncthreads();
  float scf[V], shf[V];
#pragma unroll
  for (int i = 0; i < V; ++i) { scf[i] = s_aff[c + i]; shf[i] = s_aff[p.C + c + i]; }
  long long pixb = pix0;
  for (long long e = e0; e < total;) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long eu = e + u * stride;
      if (eu < total) {
        const long long pix = pixb + u * pstep;
        float v[V], r[V];
        unpack_vec<T>(vr[u], v);
        if (res) unpack_vec<T>(rr[u], r);
#pragma unroll
        for (int i = 0; i < V; ++i) {
          float t = fmaf(v[i], scf[i], shf[i]);
          if (res) t += r[i];
          if (p.relu) t = fmaxf(t, 0.f);
          v[i] = t;
        }
        store_vec<T>(y + pix * p.ldy + c, v);
      }
    }
    e += U * stride;
    pixb += U * pstep;
    if (e < total) load_batch(e, pixb);
  }
}

__device__ __forceinline__ void lds_volatile_f4(uint32_t addr, float (&v)[4]) {
  asm volatile("ld.volatile.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(addr));
}

// per-channel sums of dy' and dy'*xhat ; dy' = relu ? (act>0 ? dy : 0) : dy.
// Lanes of a warp that own the same channel vector are folded with shuffles, warps with one shared-memory
// slot each, the block with one double atomic per channel.
// FROZEN (BatchNorm on its running statistics): dx = gamma*invstd*dy' does not depend on the sums, so the same pass also
// writes dx (and dres = dy') — BN backward in one read of dy, x (and act) and one write.
template <typename T, typename Acc, bool XMASK, bool FROZEN = false>
__device__ __forceinline__ void bn_bwd_reduce_body(const d3fk_bn_params& p, double* sred) {
  constexpr int V = Vec<T>::N;
  const int C = p.C, cvs = C / V;
  const int nwarp = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rows_per_iter = blockDim.x / cvs;
  const int cv = threadIdx.x % cvs, prow = threadIdx.x / cvs;
  const int c = cv * V;
  Acc s1[V], s2[V];
#pragma unroll
  for (int i = 0; i < V; ++i) { s1[i] = 0; s2[i] = 0; }
  constexpr bool xmask = XMASK;                      // p.relu && p.mask_from_x, resolved at launch (register budget)
  float* s_ms = reinterpret_cast<float*>(sred);      // [3][C] scale, shift, gamma*invstd — aliases the reduction slots, dead until the loop ends
  if (xmask || FROZEN) {
    for (int ch = threadIdx.x; ch < C; ch += blockDim.x) {
      if (xmask) { s_ms[ch] = p.scale[ch]; s_ms[C + ch] = p.shift[ch]; }
      if (FROZEN) s_ms[2 * C + ch] = __ldg(p.gamma + ch) * __ldg(p.invstd + ch);
    }
    __syncthreads();
  }
  const uint32_t ms_addr = (uint32_t)__cvta_generic_to_shared(s_ms + c);
  if (prow < rows_per_iter) {
    float mean[V], istd[V];
#pragma unroll
    for (int i = 0; i < V; ++i) { mean[i] = p.mean[c + i]; istd[i] = p.invstd[c + i]; }
    // mask_from_x: act = relu(x * scale + shift) was computed from exactly these x, scale, shift — its sign is recomputed
    // instead of streaming `act` a second and third time (2 of the 6 + 8 bytes per element of BN backward)
    // (scale / shift are re-read from shared memory at every use: as 2 x V registers they spill the streaming loop)
    const T* x = (const T*)p.x;
    const T* dy = (const T*)p.dy;
    const T* act = (const T*)p.act;
    constexpr int U = 2;   // independent pixel rows in flight per thread, held PACKED (4 registers per 16-byte vector)
    const long long pstride = (long long)gridDim.x * rows_per_iter;
    for (long long pix0 = (long long)blockIdx.x * rows_per_iter + prow; pix0 < p.count; pix0 += U * pstride) {
      uint4 xr[U], gr[U], ar[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long pix = pix0 + u * pstride;
        if (pix < p.count) {
          xr[u] = load_raw<T>(x + pix * p.ldx + c);
          gr[u] = load_raw<T>(dy + pix * p.lddy + c);
          if (p.relu && !xmask) ar[u] = load_raw<T>(act + pix * p.ldact + c);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (pix0 + u * pstride < p.count) {
          float xv[V], gv[V];
          unpack_vec<T>(xr[u], xv);
          unpack_vec<T>(gr[u], gv);
          if (xmask) {
#pragma unroll
            for (int i4 = 0; i4 < V; i4 += 4) {
              float kS[4], kT[4];
              lds_volatile_f4(ms_addr + 4u * i4, kS);
              lds_volatile_f4(ms_addr + 4u * (uint32_t)C + 4u * i4, kT);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const int i = i4 + j;
                float g = gv[i];
                if (!(fmaf(xv[i], kS[j], kT[j]) > 0.f)) g = 0.f;
                float xh = (xv[i] - mean[i]) * istd[i];
                s1[i] += (Acc)g;
                s2[i] += (Acc)(g * xh);
                gv[i] = g;
              }
            }
          } else {
            float av[V];
            if (p.relu) unpack_vec<T>(ar[u], av);
#pragma unroll
            for (int i = 0; i < V; ++i) {
              float g = gv[i];
              if (p.relu && !(av[i] > 0.f)) g = 0.f;
              float xh = (xv[i] - mean[i]) * istd[i];
              s1[i] += (Acc)g;
              s2[i] += (Acc)(g * xh);
              gv[i] = g;
            }
          }
          if (FROZEN) {
            const long long pix = pix0 + u * pstride;
            float o[V];
#pragma unroll
            for (int i4 = 0; i4 < V; i4 += 4) {
              float kA[4];
              lds_volatile_f4(ms_addr + 8u * (uint32_t)C + 4u * i4, kA);
#pragma unroll
              for (int j = 0; j < 4; ++j) o[i4 + j] = fmaf(kA[j], gv[i4 + j], 0.f);   // = bn_bwd_apply's A*g' + (0*(x-mean) + 0)
            }
            store_vec<T>((T*)p.dx + pix * p.lddx + c, o);
            if (p.dres) store_vec<T>((T*)p.dres + pix * p.lddres + c, gv);
          }
        }
      }
    }
  }
  if (xmask || FROZEN) __syncthreads();     // the staged scale / shift / gamma*invstd are dead: the slots below overwrite them
  // fold lanes that share cv (lane stride cvs) when a warp holds several pixel rows
  if (cvs < 32) {
#pragma unroll
    for (int i = 0; i < V; ++i) {
      for (int o = 16; o >= cvs; o >>= 1) {
        s1[i] += __shfl_xor_sync(0xffffffffu, s1[i], o);
        s2[i] += __shfl_xor_sync(0xffffffffu, s2[i], o);
      }
    }
  }
  // shared slots: cvs < 32: [warp][2][C]; cvs >= 32: a warp covers 32 consecutive channel vectors -> [warp][2][32*V]
  const int slotC = cvs < 32 ? C : 32 * V;
  if (cvs < 32) {
    if (lane < cvs) {
#pragma unroll
      for (int i = 0; i < V; ++i) {
        sred[(warp * 2 + 0) * slotC + c + i] = (double)s1[i];
        sred[(warp * 2 + 1) * slotC + c + i] = (double)s2[i];
      }
    }
  } else {
#pragma unroll
    for (int i = 0; i < V; ++i) {
      sred[(warp * 2 + 0) * slotC + lane * V + i] = (double)s1[i];
      sred[(warp * 2 + 1) * slotC + lane * V + i] = (double)s2[i];
    }
  }
  __syncthreads();
  const int groups = cvs < 32 ? 1 : cvs / 32;   // warps w, w+groups, ... hold the same channel range
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) {
    const int which = i / C, ch = i - which * C;
    const int grp = cvs < 32 ? 0 : ch / slotC;
    const int within = cvs < 32 ? ch : ch % slotC;
    double a = 0;
    for (int w = grp; w < nwarp; w += groups) a += sred[(w * 2 + which) * slotC + within];
    atomicAdd(&p.bstats[which * C + ch], a);
  }
}
template <typename T, typename Acc, bool XMASK>
__global__ void __launch_bounds__(256, BN_BWD_OCC(T)) bn_bwd_reduce_kernel(d3fk_bn_params p) {
  pdl_enter();
  extern __shared__ double sred_dyn[];  // [warps][2][C]
  bn_bwd_reduce_body<T, Acc, XMASK>(p, sred_dyn);
}

// frozen BN backward, one pass: dx (and dres) written, sum(dy') / sum(dy' * xhat) accumulated; bn_bwd_finalize writes dgamma / dbeta
// (two blocks per SM on the bf16 engine: the dx / dres stores need the registers the three-block budget of the reduce kernel lacks)
template <typename T, typename Acc, bool XMASK>
__global__ void __launch_bounds__(256, sizeof(T) == 2 ? 2 : 1) bn_bwd_frozen_kernel(d3fk_bn_params p) {
  pdl_enter();
  extern __shared__ double sred_dyn[];  // [warps][2][C]
  bn_bwd_reduce_body<T, Acc, XMASK, true>(p, sred_dyn);
}

__global__ void bn_bwd_finalize_kernel(d3fk_bn_params p) {
  pdl_enter();
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= p.C) return;
  double n = (double)p.count;
  double s1 = p.bstats[c], s2 = p.bstats[p.C + c];
  if (p.dbeta) p.dbeta[c] = (float)s1;
  if (p.dgamma) p.dgamma[c] = (float)s2;
  if (!p.coef) return;
  p.coef[c] = p.gamma[c] * p.invstd[c];
  p.coef[p.C + c] = (float)(s1 / n);
  p.coef[2 * p.C + c] = (float)(s2 / n);
}


// dx = c0*(dy' - c1 - xhat*c2), c0 = gamma*invstd, c1 = sum(dy')/n, c2 = sum(dy'*xhat)/n; optionally dres = dy'.
// The coefficients are derived in-kernel from the reduction sums; the first C/V threads of block 0 also write
// dgamma / dbeta (no separate finalize launch).
template <typename T, bool XMASK>
__device__ __forceinline__ void bn_bwd_apply_body(const d3fk_bn_params& p, float* s_k) {
  constexpr int V = Vec<T>::N;
  const int cvs = p.C / V;
  const long long total = p.count * cvs;
  const T* x = (const T*)p.x;
  const T* dy = (const T*)p.dy;
  const T* act = (const T*)p.act;
  T* dx = (T*)p.dx;
  T* dres = (T*)p.dres;
  const long long e0 = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const int c = (int)(e0 % cvs) * V;
  // s_k: [4][C]: A = gamma*invstd, Bm = -A*invstd*sum(dy'*xhat)/n, C1 = -A*sum(dy')/n, mean — derived once per block (L2
  // loads: the sums were produced by atomics), so that dx = A*dy' + Bm*(x - mean) + C1.  The coefficients stay in shared
  // memory and are re-read (volatile 16-byte loads, warp-broadcast) at every use: as 5 x V registers per thread they cost a
  // third of the register file and one of the three resident blocks.
  for (int ch = threadIdx.x; ch < p.C; ch += blockDim.x) {
    const double n = (double)p.count;
    const double s1 = __ldcg(p.bstats + ch), s2 = __ldcg(p.bstats + p.C + ch);
    const float is = __ldg(p.invstd + ch);
    const float A = __ldg(p.gamma + ch) * is;
    s_k[ch] = A;
    // frozen (running statistics): the normalisation is a constant affine map, dx = A*dy'
    s_k[p.C + ch] = p.frozen ? 0.f : -A * is * (float)(s2 / n);
    s_k[2 * p.C + ch] = p.frozen ? 0.f : -A * (float)(s1 / n);
    s_k[3 * p.C + ch] = __ldg(p.mean + ch);
    if (XMASK) {
      s_k[4 * p.C + ch] = p.scale[ch];
      s_k[5 * p.C + ch] = p.shift[ch];
    }
    if (blockIdx.x == 0) {
      if (p.dbeta) p.dbeta[ch] = (float)s1;
      if (p.dgamma) p.dgamma[ch] = (float)s2;
    }
  }
  __syncthreads();
  const uint32_t sk_addr = (uint32_t)__cvta_generic_to_shared(s_k + c);
  const uint32_t sk_pitch = (uint32_t)p.C * 4u;
  constexpr int U = 2;   // independent pixel vectors in flight per thread (3 loads each), held packed until used
  constexpr bool xmask = XMASK;
  // Walk the tensor BACKWARDS: the reduction pass that ran just before streamed x, dy and act front to back, so their
  // tails are what the 126 MB L2 still holds.
  const long long last_pix = p.count - 1;
  const long long pstep = stride / cvs;          // stride is a multiple of cvs: element e0 + k * stride is pixel e0 / cvs + k * pstep
  long long pixb = last_pix - e0 / cvs;
  for (long long e = e0; e < total; e += U * stride, pixb -= U * pstep) {
    uint4 xr[U], gr[U], ar[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long eu = e + u * stride;
      if (eu < total) {
        const long long pix = pixb - u * pstep;
        xr[u] = load_raw<T>(x + pix * p.ldx + c);
        gr[u] = load_raw<T>(dy + pix * p.lddy + c);
        if (p.relu && !xmask) ar[u] = load_raw<T>(act + pix * p.ldact + c);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long eu = e + u * stride;
      if (eu < total) {
        const long long pix = pixb - u * pstep;
        float xv[V], gv[V], av[V], o[V];
        unpack_vec<T>(xr[u], xv);
        unpack_vec<T>(gr[u], gv);
        if (p.relu && !xmask) unpack_vec<T>(ar[u], av);
#pragma unroll
        for (int i4 = 0; i4 < V; i4 += 4) {
          float kA[4], kB[4], kC[4], kM[4];
          lds_volatile_f4(sk_addr + 4u * i4, kA);
          lds_volatile_f4(sk_addr + sk_pitch + 4u * i4, kB);
          lds_volatile_f4(sk_addr + 2u * sk_pitch + 4u * i4, kC);
          lds_volatile_f4(sk_addr + 3u * sk_pitch + 4u * i4, kM);
          if (xmask) {
            float kS[4], kT[4];
            lds_volatile_f4(sk_addr + 4u * sk_pitch + 4u * i4, kS);
            lds_volatile_f4(sk_addr + 5u * sk_pitch + 4u * i4, kT);
#pragma unroll
            for (int j = 0; j < 4; ++j) av[i4 + j] = fmaf(xv[i4 + j], kS[j], kT[j]);
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int i = i4 + j;
            float g = gv[i];
            if (p.relu && !(av[i] > 0.f)) g = 0.f;
            gv[i] = g;
            o[i] = fmaf(kA[j], g, fmaf(kB[j], xv[i] - kM[j], kC[j]));
          }
        }
        store_vec<T>(dx + pix * p.lddx + c, o);
        if (dres) store_vec<T>(dres + pix * p.lddres + c, gv);
      }
    }
  }
}

template <typename T, bool XMASK>
__global__ void __launch_bounds__(256, BN_BWD_OCC(T)) bn_bwd_apply_kernel(d3fk_bn_params p) {
  pdl_enter();
  extern __shared__ float s_k_dyn[];
  bn_bwd_apply_body<T, XMASK>(p, s_k_dyn);
}

// BN backward in ONE launch for a co-resident grid: reduction, grid barrier, apply (the tensors of the deep layers are a
// few MB — the second read comes from L2 and a kernel boundary costs more than the barrier).
template <typename T, typename Acc, bool XMASK>
__global__ void __launch_bounds__(256, 2) bn_bwd_kernel(d3fk_bn_params p, int* errflag) {
  pdl_enter();
  extern __shared__ double smem_bwd[];
  bn_bwd_reduce_body<T, Acc, XMASK>(p, smem_bwd);
  __syncthreads();
  if (threadIdx.x == 0) grid_barrier_arrive_wait(p.barrier, gridDim.x, errflag);
  __syncthreads();
  bn_bwd_apply_body<T, XMASK>(p, reinterpret_cast<float*>(smem_bwd));
}

// element index -> (pixel, channel vector, w, h, n) of a [n][h][w][cvs] walk.  32-bit arithmetic whenever the index fits
// (always, at the sizes this path sees): five 64-bit divisions per 16-byte vector made the pool kernels issue-bound.
__device__ __forceinline__ void split_index(long long e, int cvs, int W, int H, long long& pix, int& cv, int& w, int& h, int& n) {
  if (e < 0x7fffffffLL) {
    const unsigned ue = (unsigned)e, up = ue / (unsigned)cvs;
    cv = (int)(ue - up * (unsigned)cvs);
    const unsigned t = up / (unsigned)W;
    w = (int)(up - t * (unsigned)W);
    const unsigned un = t / (unsigned)H;
    h = (int)(t - un * (unsigned)H);
    n = (int)un;
    pix = (long long)up;
  } else {
    pix = e / cvs;
    cv = (int)(e - pix * cvs);
    w = (int)(pix % W);
    const long long t = pix / W;
    h = (int)(t % H);
    n = (int)(t / H);
  }
}

// ---------------------------------------------------------------------------------------------
// MaxPool2d(kernel 3, stride 2, pad 1): first-max tie-break in window scan order (ATen semantics)
template <typename T>
__global__ void maxpool_fwd_kernel(d3fk_pool_params p) {
  pdl_enter();
  constexpr int V = Vec<T>::N;
  const int Ho = p.H / 2, Wo = p.W / 2, cvs = p.C / V;
  const long long total = (long long)p.B * Ho * Wo * cvs;
  const T* x = (const T*)p.x;
  T* y = (T*)p.y;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    long long pix;
    int c, wo, ho, n;
    split_index(e, cvs, Wo, Ho, pix, c, wo, ho, n);
    c *= V;
    float best[V];
    unsigned char bi[V];
#pragma unroll
    for (int i = 0; i < V; ++i) { best[i] = -INFINITY; bi[i] = 0; }
    // all nine 16-byte loads are issued before the first compare (out-of-image taps load a clamped, valid address and are
    // skipped by predicate): nine independent requests in flight per thread instead of a branchy load-compare chain
    uint4 raw[9];
    bool ok[9];
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
      const int h = 2 * ho - 1 + kh;
      const bool hok = (unsigned)h < (unsigned)p.H;
      const int hc = hok ? h : 2 * ho;
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int w = 2 * wo - 1 + kw;
        const bool wok = (unsigned)w < (unsigned)p.W;
        const int wc = wok ? w : 2 * wo;
        ok[kh * 3 + kw] = hok && wok;
        raw[kh * 3 + kw] = *reinterpret_cast<const uint4*>(x + ((long long)(n * p.H + hc) * p.W + wc) * p.ldx + c);
      }
    }
    bool first = true;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      if (!ok[t]) continue;
      const T* e8 = reinterpret_cast<const T*>(&raw[t]);
#pragma unroll
      for (int i = 0; i < V; ++i) {
        const float v = to_f<T>(e8[i]);
        if (first || v > best[i] || v != v) { best[i] = v; bi[i] = (unsigned char)t; }
      }
      first = false;
    }
    store_vec<T>(y + pix * p.ldy + c, best);
    if (p.idx) {
      unsigned long long pk = 0ull;          // one 8-byte (V = 8) / 4-byte (V = 4) store instead of V byte stores
#pragma unroll
      for (int i = 0; i < V; ++i) pk |= (unsigned long long)bi[i] << (8 * i);
      if (V == 8) *reinterpret_cast<unsigned long long*>(p.idx + pix * p.C + c) = pk;
      else *reinterpret_cast<unsigned int*>(p.idx + pix * p.C + c) = (unsigned int)pk;
    }
  }
}

// One thread per 2x2 block of dx (rows 2a, 2a+1; columns 2b, 2b+1) and channel vector: the four dx pixels are covered by
// the pooled windows (a .. a+1) x (b .. b+1) only, so 4 dy + 4 index loads serve 4 outputs (the pixel-per-thread form loaded
// up to 4 + 4 per output and was L2-traffic bound: 45 us for the stem's 16.8 M elements).
template <typename T>
__global__ void __launch_bounds__(256) maxpool_bwd_kernel(d3fk_pool_params p) {
  pdl_enter();
  constexpr int V = Vec<T>::N;
  const int Ho = p.H / 2, Wo = p.W / 2, cvs = p.C / V;
  const long long total = (long long)p.B * Ho * Wo * cvs;
  const T* dy = (const T*)p.dy;
  T* dx = (T*)p.dx;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    long long blk;
    int c, b, a, n;
    split_index(e, cvs, Wo, Ho, blk, c, b, a, n);
    c *= V;
    float d[2][2][V];
    unsigned long long ipk[2][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        ipk[i][j] = ~0ull;                                   // no tap matches: the window is outside the pooled map
        if (a + i < Ho && b + j < Wo) {
          const long long op = (long long)(n * Ho + a + i) * Wo + b + j;
          load_vec<T>(dy + op * p.lddy + c, d[i][j]);
          // the V tap indices of this channel vector in ONE load (V = 8: 8 bytes, V = 4: 4 bytes) instead of V byte loads
          if (V == 8) ipk[i][j] = __ldg(reinterpret_cast<const unsigned long long*>(p.idx + op * p.C + c));
          else ipk[i][j] = (unsigned long long)__ldg(reinterpret_cast<const unsigned int*>(p.idx + op * p.C + c)) | 0xFFFFFFFF00000000ull;
        } else {
#pragma unroll
          for (int k = 0; k < V; ++k) d[i][j][k] = 0.f;
        }
      }
#pragma unroll
    for (int di = 0; di < 2; ++di)
#pragma unroll
      for (int dj = 0; dj < 2; ++dj) {
        const long long pix = ((long long)n * p.H + 2 * a + di) * p.W + 2 * b + dj;
        float g[V];
#pragma unroll
        for (int k = 0; k < V; ++k) g[k] = 0.f;
        if (p.accumulate) load_vec<T>(dx + pix * p.lddx + c, g);
        // pixel (2a + di, 2b + dj) lies in window (a + i, b + j) for i <= di, j <= dj, at tap (di - 2i + 1, dj - 2j + 1)
#pragma unroll
        for (int i = 0; i <= di; ++i)
#pragma unroll
          for (int j = 0; j <= dj; ++j) {
            const int tap = (di - 2 * i + 1) * 3 + (dj - 2 * j + 1);
#pragma unroll
            for (int k = 0; k < V; ++k)
              if ((int)((ipk[i][j] >> (8 * k)) & 0xFFull) == tap) g[k] += d[i][j][k];
          }
        store_vec<T>(dx + pix * p.lddx + c, g);
      }
  }
}

// backward of nearest 2x upsample: dx[n,h,w,c] = sum of the 2x2 block of dy (H,W = low-res extent)
template <typename T>
__global__ void sumpool2_kernel(d3fk_pool_params p) {
  pdl_enter();
  constexpr int V = Vec<T>::N;
  const int cvs = p.C / V;
  const long long total = (long long)p.B * p.H * p.W * cvs;
  const T* dy = (const T*)p.dy;
  T* dx = (T*)p.dx;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    long long pix;
    int c, w, h, n;
    split_index(e, cvs, p.W, p.H, pix, c, w, h, n);
    c *= V;
    float g[V];
#pragma unroll
    for (int i = 0; i < V; ++i) g[i] = 0.f;
    if (p.accumulate) load_vec<T>(dx + pix * p.lddx + c, g);
#pragma unroll
    for (int dh = 0; dh < 2; ++dh)
#pragma unroll
      for (int dw = 0; dw < 2; ++dw) {
        float d[V];
        load_vec<T>(dy + ((long long)(n * 2 * p.H + 2 * h + dh) * (2 * p.W) + 2 * w + dw) * p.lddy + c, d);
#pragma unroll
        for (int i = 0; i < V; ++i) g[i] += d[i];
      }
    store_vec<T>(dx + pix * p.lddx + c, g);
  }
}

// nearest 2x upsample of src0 concatenated with src1 along channels (16-byte vectors; C's are multiples of 8 / 4)
template <typename T>
__global__ void __launch_bounds__(256) upcat_kernel(d3fk_upcat_params p) {
  pdl_enter();
  // One block per output image row: the (n, h) split is done once per block and the per-vector index is one 32-bit
  // division — the element-indexed form spent ~250 instructions (five 64-bit divisions) per 16-byte vector and was
  // issue-bound at 55 % of the HBM rate.
  constexpr int V = Vec<T>::N;
  const int cv0 = p.c0 / V, cvs = (p.c0 + p.c1) / V;
  const uint4* s0 = (const uint4*)p.src0;
  const uint4* s1 = (const uint4*)p.src1;
  uint4* out = (uint4*)p.out;
  const int Hs = p.H >> 1, Ws = p.W >> 1;
  const int per_row = p.W * cvs;
  const int ld0v = p.ld0 / V, ld1v = p.ld1 / V, ldov = p.ldo / V;
  for (long long r = blockIdx.x; r < (long long)p.B * p.H; r += gridDim.x) {
    const int n = (int)(r / p.H), h = (int)(r - (long long)n * p.H);
    const uint4* row0 = s0 + ((long long)(n * Hs + (h >> 1)) * Ws) * ld0v;
    const uint4* row1 = s1 + (r * p.W) * ld1v;
    uint4* orow = out + (r * p.W) * ldov;
    for (int i = threadIdx.x; i < per_row; i += blockDim.x) {
      const int w = i / cvs, cv = i - w * cvs;
      uint4 v;
      if (cv < cv0) v = __ldg(row0 + (long long)(w >> 1) * ld0v + cv);
      else v = __ldg(row1 + (long long)w * ld1v + (cv - cv0));
      orow[(long long)w * ldov + cv] = v;
    }
  }
}

// out[c] += sum over pixels x[pix*ld + c], c < C <= 8
template <typename T>
__global__ void chansum_kernel(d3fk_chansum_params p) {
  pdl_enter();
  constexpr int V = Vec<T>::N;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  const T* x = (const T*)p.x;
  for (long long pix = blockIdx.x * (long long)blockDim.x + threadIdx.x; pix < p.count; pix += (long long)gridDim.x * blockDim.x) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.f;
    load_vec<T>(x + pix * p.ld, v);
    if (V == 4 && p.C > 4) load_vec<T>(x + pix * p.ld + 4, v + 4);
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] += v[i];
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float a = acc[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if ((threadIdx.x & 31) == 0 && i < p.C) atomicAdd(p.out + i, a);
  }
}

// ---------------------------------------------------------------------------------------------
// q_sample: out = sqrt(1-r_b) x + sqrt(r_b) eps   (d3f/train_denoiser/lit_module.py:128-153)
// sqrt(1-r) x + sqrt(r) n with a FIXED rounding order (one product rounded, then one fused multiply-add): q_sample and the
// fused affine + q_sample kernel must agree bit for bit, whatever contraction the compiler would pick in each.
__device__ __forceinline__ float blend1(float a, float x, float s, float n) { return __fmaf_rn(a, x, __fmul_rn(s, n)); }

// blockIdx.y = sample: the noise ratio r_b (one Philox draw, one log, two square roots) is formed once per block, not once
// per 4 elements; the Philox counter of the element noise is still the global vector index, so results are unchanged.
__global__ void __launch_bounds__(256) qsample_kernel(d3fk_qsample_params p) {
  pdl_enter();
  const int vec_per_sample = p.chw / 4;
  const int b = blockIdx.y;
  __shared__ float s_coef[2];
  if (threadIdx.x == 0) {
    float r;
    if (p.fixed_r >= 0.f) {
      r = p.fixed_r;
    } else {
      const float cexp = expf(-p.lam);     // once per block: the accurate form
      float y;
      if (p.y) y = __ldg(p.y + b);
      else {
        uint4 u = philox4x32_10(make_uint4((uint32_t)b, 0u, (uint32_t)p.offset, 0x9E3779B9u),
                                make_uint2((uint32_t)p.seed, (uint32_t)(p.seed >> 32)));
        y = (float)(u.x >> 8) * (1.0f / 16777216.0f);  // U[0,1) like torch.rand
      }
      r = (1.0f / p.lam) * logf(1.0f / (y * (1.0f - cexp) + cexp));
      r = fminf(fmaxf(r, 0.f), 1.f);   // y == 0 can round to 1 + ulp: sqrtf(1 - r) would be NaN for the whole sample
    }
    s_coef[0] = sqrtf(1.0f - r);
    s_coef[1] = sqrtf(r);
    if (p.r_out && blockIdx.x == 0) p.r_out[b] = r;
  }
  __syncthreads();
  const float a = s_coef[0], s = s_coef[1];
  const long long base = (long long)b * vec_per_sample;
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < vec_per_sample; v += gridDim.x * blockDim.x) {
    const long long i = base + v;
    float4 x = __ldg(reinterpret_cast<const float4*>(p.x) + i);
    float4 n;
    if (p.noise) n = __ldg(reinterpret_cast<const float4*>(p.noise) + i);
    else n = philox_normal4(p.seed, (uint64_t)i, p.offset);
    float4 o = make_float4(blend1(a, x.x, s, n.x), blend1(a, x.y, s, n.y), blend1(a, x.z, s, n.z), blend1(a, x.w, s, n.w));
    reinterpret_cast<float4*>(p.out)[i] = o;
    if (p.noise_out) reinterpret_cast<float4*>(p.noise_out)[i] = n;
  }
}

// Random affine warp (bilinear, zero padding) fused with q_sample.  blockIdx.y = sample; a thread owns 4 consecutive
// elements of the NCHW sample (W % 4 == 0: the same image row and channel), i.e. exactly the vector qsample_kernel owns,
// so the Philox counters — and therefore the noise — are those of q_sample applied to the augmented image.
__global__ void __launch_bounds__(256) affine_qsample_kernel(d3fk_affine_qsample_params p) {
  pdl_enter();
  const int hw = p.H * p.W;
  const int vec_per_sample = p.C * hw / 4;
  const int b = blockIdx.y;
  __shared__ float s_coef[2];
  __shared__ float s_m[6];
  if (threadIdx.x < 6) s_m[threadIdx.x] = __ldg(p.minv + 6 * b + threadIdx.x);
  if (threadIdx.x == 32) {
    float r;
    if (p.fixed_r >= 0.f) {
      r = p.fixed_r;
    } else {
      const float cexp = expf(-p.lam);     // once per block: the accurate form
      float y;
      if (p.y) y = __ldg(p.y + b);
      else {
        uint4 u = philox4x32_10(make_uint4((uint32_t)b, 0u, (uint32_t)p.offset, 0x9E3779B9u),
                                make_uint2((uint32_t)p.seed, (uint32_t)(p.seed >> 32)));
        y = (float)(u.x >> 8) * (1.0f / 16777216.0f);
      }
      r = (1.0f / p.lam) * logf(1.0f / (y * (1.0f - cexp) + cexp));
      r = fminf(fmaxf(r, 0.f), 1.f);   // y == 0 can round to 1 + ulp: sqrtf(1 - r) would be NaN for the whole sample
    }
    s_coef[0] = sqrtf(1.0f - r);
    s_coef[1] = sqrtf(r);
    if (p.r_out && blockIdx.x == 0) p.r_out[b] = r;
  }
  __syncthreads();
  const float a = s_coef[0], s = s_coef[1];
  const float m0 = s_m[0], m1 = s_m[1], m2 = s_m[2], m3 = s_m[3], m4 = s_m[4], m5 = s_m[5];
  const long long base = (long long)b * vec_per_sample;
  const float* xs = p.x + (long long)b * p.C * hw;
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < vec_per_sample; v += gridDim.x * blockDim.x) {
    const int e = 4 * v;                  // element within the sample: (c, oy, ox .. ox+3)
    const int c = e / hw;
    const int pix = e - c * hw;
    const int oy = pix / p.W, ox = pix - oy * p.W;
    const float* plane = xs + (long long)c * hw;
    float g[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float fx = (float)(ox + j), fy = (float)oy;
      const float sx = fmaf(m0, fx, fmaf(m1, fy, m2));
      const float sy = fmaf(m3, fx, fmaf(m4, fy, m5));
      const float x0f = floorf(sx), y0f = floorf(sy);
      const float wx1 = sx - x0f, wy1 = sy - y0f, wx0 = 1.f - wx1, wy0 = 1.f - wy1;
      const int x0 = (int)x0f, y0 = (int)y0f;
      const bool in_x0 = (unsigned)x0 < (unsigned)p.W, in_x1 = (unsigned)(x0 + 1) < (unsigned)p.W;
      const bool in_y0 = (unsigned)y0 < (unsigned)p.H, in_y1 = (unsigned)(y0 + 1) < (unsigned)p.H;
      const float v00 = (in_x0 && in_y0) ? __ldg(plane + y0 * p.W + x0) : 0.f;
      const float v01 = (in_x1 && in_y0) ? __ldg(plane + y0 * p.W + x0 + 1) : 0.f;
      const float v10 = (in_x0 && in_y1) ? __ldg(plane + (y0 + 1) * p.W + x0) : 0.f;
      const float v11 = (in_x1 && in_y1) ? __ldg(plane + (y0 + 1) * p.W + x0 + 1) : 0.f;
      g[j] = wy0 * (wx0 * v00 + wx1 * v01) + wy1 * (wx0 * v10 + wx1 * v11);
    }
    const long long i = base + v;
    float4 n;
    if (p.noise) n = __ldg(reinterpret_cast<const float4*>(p.noise) + i);
    else n = philox_normal4(p.seed, (uint64_t)i, p.offset);
    if (p.out_aug) reinterpret_cast<float4*>(p.out_aug)[i] = make_float4(g[0], g[1], g[2], g[3]);
    reinterpret_cast<float4*>(p.out_noisy)[i] =
        make_float4(blend1(a, g[0], s, n.x), blend1(a, g[1], s, n.y), blend1(a, g[2], s, n.z), blend1(a, g[3], s, n.w));
  }
}

// posterior: x = k_xi*x + k_x0*x0_hat + sigma*z.  The rounding is spelled out (the product k_x0*h rounded, then one fma
// each for the x and z terms) so the plain and the masked kernel agree bit for bit whatever contraction the compiler would
// pick in each; it is the contraction the plain kernel has always compiled to.
__device__ __forceinline__ float posterior1(float k_xi, float x, float k_x0, float h) {
  return __fmaf_rn(k_xi, x, __fmul_rn(k_x0, h));
}
__device__ __forceinline__ float4 posterior4(float k_xi, float4 x, float k_x0, float4 h) {
  return make_float4(posterior1(k_xi, x.x, k_x0, h.x), posterior1(k_xi, x.y, k_x0, h.y), posterior1(k_xi, x.z, k_x0, h.z),
                     posterior1(k_xi, x.w, k_x0, h.w));
}
__device__ __forceinline__ void posterior_add_noise4(float4& o, float sigma, float4 z) {
  o.x = __fmaf_rn(sigma, z.x, o.x); o.y = __fmaf_rn(sigma, z.y, o.y);
  o.z = __fmaf_rn(sigma, z.z, o.z); o.w = __fmaf_rn(sigma, z.w, o.w);
}

struct PosteriorCoefs {
  float k_xi, k_x0, sigma, r_prev;
  uint64_t off;
};
__device__ __forceinline__ PosteriorCoefs posterior_coefs(const d3fk_posterior_params& p) {
  PosteriorCoefs c{p.k_xi, p.k_x0, p.sigma, p.r_prev, p.offset};
  if (p.coef_table) {
    int s = *p.step;
    c.k_xi = p.coef_table[4 * s];
    c.k_x0 = p.coef_table[4 * s + 1];
    c.sigma = p.coef_table[4 * s + 2];
    c.r_prev = p.coef_table[4 * s + 3];
    c.off += (uint64_t)s;
  }
  return c;
}

__global__ void posterior_kernel(d3fk_posterior_params p) {
  pdl_enter();
  const PosteriorCoefs c = posterior_coefs(p);
  const long long nvec = p.n / 4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    float4 x = reinterpret_cast<const float4*>(p.x)[i];
    float4 h = __ldg(reinterpret_cast<const float4*>(p.x0_hat) + i);
    float4 o = posterior4(c.k_xi, x, c.k_x0, h);
    if (c.sigma != 0.f) {
      float4 z;
      if (p.z) z = __ldg(reinterpret_cast<const float4*>(p.z) + i);
      else z = philox_normal4(p.seed, (uint64_t)i, c.off);
      posterior_add_noise4(o, c.sigma, z);
    }
    reinterpret_cast<float4*>(p.x)[i] = o;
  }
}

__device__ __forceinline__ float composite1(float m, float post, float known) {
  return __fmaf_rn(m, post, __fmul_rn(1.f - m, known));
}
__device__ __forceinline__ float clamp01(float m) { return fminf(fmaxf(m, 0.f), 1.f); }   // NaN -> 0 (keep)

// Masked posterior (replacement inpainting): x = m*post + (1 - m)*known, known = src noised to r_prev (d3fk.h).
// blockIdx.y = sample; a thread owns the 4-element vector i = b*chw/4 + v of one channel row, exactly the vector
// posterior_kernel owns (same z counter), and reads its 4 pixels' mask (the C channels of a pixel read the same mask
// vector; after the first it comes from L2).  A vector whose 4 mask values are all 1 reads no src and draws no n; all 0
// reads no x / x0_hat and draws no z — with a hard mask each pixel costs the bytes of only one of the two updates.
__global__ void __launch_bounds__(256) posterior_masked_kernel(d3fk_posterior_params p) {
  pdl_enter();
  const PosteriorCoefs c = posterior_coefs(p);
  const float a = sqrtf(1.f - c.r_prev), s = sqrtf(c.r_prev);
  const int b = blockIdx.y;
  const unsigned vpp = (unsigned)p.hw / 4u, vps = (unsigned)p.chw / 4u;
  const long long base = (long long)b * vps;
  const float4* mask = reinterpret_cast<const float4*>(p.mask) + (long long)b * vpp;
  for (unsigned v = blockIdx.x * blockDim.x + threadIdx.x; v < vps; v += gridDim.x * blockDim.x) {
    float4 m = __ldg(mask + v % vpp);
    m = make_float4(clamp01(m.x), clamp01(m.y), clamp01(m.z), clamp01(m.w));
    const bool all1 = m.x == 1.f && m.y == 1.f && m.z == 1.f && m.w == 1.f;
    const bool all0 = m.x == 0.f && m.y == 0.f && m.z == 0.f && m.w == 0.f;
    const long long i = base + v;
    float4 post = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!all0) {
      float4 x = reinterpret_cast<const float4*>(p.x)[i];
      float4 h = __ldg(reinterpret_cast<const float4*>(p.x0_hat) + i);
      post = posterior4(c.k_xi, x, c.k_x0, h);
      if (c.sigma != 0.f) {
        float4 z;
        if (p.z) z = __ldg(reinterpret_cast<const float4*>(p.z) + i);
        else z = philox_normal4(p.seed, (uint64_t)i, c.off);
        posterior_add_noise4(post, c.sigma, z);
      }
    }
    float4 known = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!all1) {
      float4 n = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c.r_prev != 0.f) {
        if (p.known_noise) n = __ldg(reinterpret_cast<const float4*>(p.known_noise) + i);
        else n = philox_normal4(p.seed, (uint64_t)i | (1ull << 63), c.off);
      }
      float4 x = __ldg(reinterpret_cast<const float4*>(p.src) + i);
      known = make_float4(blend1(a, x.x, s, n.x), blend1(a, x.y, s, n.y), blend1(a, x.z, s, n.z), blend1(a, x.w, s, n.w));
    }
    reinterpret_cast<float4*>(p.x)[i] = make_float4(composite1(m.x, post.x, known.x), composite1(m.y, post.y, known.y),
                                                    composite1(m.z, post.z, known.z), composite1(m.w, post.w, known.w));
  }
}

// Second-order multistep (DPM-Solver++ 2M) posterior, d3fk.h: D = x0_hat + c*(x0_hat - x0_prev) stands in for x0_hat in
// the update above, and x0_prev <- x0_hat for the next step.  With c == 0 x0_prev is only written (D is x0_hat itself),
// so the result is the posterior kernel's bit for bit and a step needs 16 B/element; with c != 0, 20 B/element.
static_assert(sizeof(d3fk_posterior_2m_params) == 128 && offsetof(d3fk_posterior_2m_params, x0_prev) == 112 &&
              offsetof(d3fk_posterior_2m_params, c) == 120 && sizeof(d3fk_op) == 480, "d3fk_posterior_2m_params ABI");
struct Posterior2mCoefs {
  PosteriorCoefs b;
  float c;
};
__device__ __forceinline__ Posterior2mCoefs posterior_2m_coefs(const d3fk_posterior_2m_params& p) {
  const d3fk_posterior_params& q = p.base;
  Posterior2mCoefs c{{q.k_xi, q.k_x0, q.sigma, q.r_prev, q.offset}, p.c};
  if (q.coef_table) {
    const int s = *q.step;
    const float* row = q.coef_table + 5 * s;
    c.b.k_xi = row[0];
    c.b.k_x0 = row[1];
    c.b.sigma = row[2];
    c.b.r_prev = row[3];
    c.c = row[4];
    c.b.off += (uint64_t)s;
  }
  return c;
}
// D = fma(c, h - p, h), the difference rounded first.
__device__ __forceinline__ float4 multistep4(float c, float4 h, float4 p) {
  return make_float4(__fmaf_rn(c, __fsub_rn(h.x, p.x), h.x), __fmaf_rn(c, __fsub_rn(h.y, p.y), h.y),
                     __fmaf_rn(c, __fsub_rn(h.z, p.z), h.z), __fmaf_rn(c, __fsub_rn(h.w, p.w), h.w));
}

__global__ void posterior_2m_kernel(d3fk_posterior_2m_params p) {
  pdl_enter();
  const Posterior2mCoefs c = posterior_2m_coefs(p);
  const d3fk_posterior_params& q = p.base;
  float4* prev = reinterpret_cast<float4*>(p.x0_prev);
  const long long nvec = q.n / 4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    float4 x = reinterpret_cast<const float4*>(q.x)[i];
    float4 h = __ldg(reinterpret_cast<const float4*>(q.x0_hat) + i);
    float4 d = h;
    if (c.c != 0.f) d = multistep4(c.c, h, prev[i]);
    prev[i] = h;
    float4 o = posterior4(c.b.k_xi, x, c.b.k_x0, d);
    if (c.b.sigma != 0.f) {
      float4 z;
      if (q.z) z = __ldg(reinterpret_cast<const float4*>(q.z) + i);
      else z = philox_normal4(q.seed, (uint64_t)i, c.b.off);
      posterior_add_noise4(o, c.b.sigma, z);
    }
    reinterpret_cast<float4*>(q.x)[i] = o;
  }
}

// Masked form: posterior_masked_kernel with D for x0_hat; all-0 mask vectors read no x0_hat and leave x0_prev as it is.
__global__ void __launch_bounds__(256) posterior_2m_masked_kernel(d3fk_posterior_2m_params p) {
  pdl_enter();
  const Posterior2mCoefs cc = posterior_2m_coefs(p);
  const PosteriorCoefs& c = cc.b;
  const d3fk_posterior_params& q = p.base;
  float4* prev = reinterpret_cast<float4*>(p.x0_prev);
  const float a = sqrtf(1.f - c.r_prev), s = sqrtf(c.r_prev);
  const int b = blockIdx.y;
  const unsigned vpp = (unsigned)q.hw / 4u, vps = (unsigned)q.chw / 4u;
  const long long base = (long long)b * vps;
  const float4* mask = reinterpret_cast<const float4*>(q.mask) + (long long)b * vpp;
  for (unsigned v = blockIdx.x * blockDim.x + threadIdx.x; v < vps; v += gridDim.x * blockDim.x) {
    float4 m = __ldg(mask + v % vpp);
    m = make_float4(clamp01(m.x), clamp01(m.y), clamp01(m.z), clamp01(m.w));
    const bool all1 = m.x == 1.f && m.y == 1.f && m.z == 1.f && m.w == 1.f;
    const bool all0 = m.x == 0.f && m.y == 0.f && m.z == 0.f && m.w == 0.f;
    const long long i = base + v;
    float4 post = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!all0) {
      float4 x = reinterpret_cast<const float4*>(q.x)[i];
      float4 h = __ldg(reinterpret_cast<const float4*>(q.x0_hat) + i);
      float4 d = h;
      if (cc.c != 0.f) d = multistep4(cc.c, h, prev[i]);
      prev[i] = h;
      post = posterior4(c.k_xi, x, c.k_x0, d);
      if (c.sigma != 0.f) {
        float4 z;
        if (q.z) z = __ldg(reinterpret_cast<const float4*>(q.z) + i);
        else z = philox_normal4(q.seed, (uint64_t)i, c.off);
        posterior_add_noise4(post, c.sigma, z);
      }
    }
    float4 known = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!all1) {
      float4 n = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c.r_prev != 0.f) {
        if (q.known_noise) n = __ldg(reinterpret_cast<const float4*>(q.known_noise) + i);
        else n = philox_normal4(q.seed, (uint64_t)i | (1ull << 63), c.off);
      }
      float4 x = __ldg(reinterpret_cast<const float4*>(q.src) + i);
      known = make_float4(blend1(a, x.x, s, n.x), blend1(a, x.y, s, n.y), blend1(a, x.z, s, n.z), blend1(a, x.w, s, n.w));
    }
    reinterpret_cast<float4*>(q.x)[i] = make_float4(composite1(m.x, post.x, known.x), composite1(m.y, post.y, known.y),
                                                    composite1(m.z, post.z, known.z), composite1(m.w, post.w, known.w));
  }
}

__global__ void inc_kernel(int* p) {
  pdl_enter(); *p += 1; }

// One launch packs every convolution's weights (fp32 OIHW master -> K-major forward / dgrad operands).
// A block owns a 32 (cout) x 32 (cin) x taps sub-tensor of one layer: coalesced fp32 reads of the 32 rows of
// (32 cin x taps) contiguous floats into a padded shared tile, then 32-channel contiguous writes in both layouts:
//   w_fwd  [Cout][tap][cin_pad]  (lanes = cin)      w_dgrad [Cin][tap][cout_pad]  (lanes = cout)
// blk0 of each table entry is the first block of that layer; padding columns are never written (buffers start zeroed).
constexpr int PK_T = 32;
constexpr int PK_MAXCOL = 32 * 9;          // 3x3 with a full cin block; the 7x7 stem has 3 x 49 = 147 columns
template <typename T>
__global__ void __launch_bounds__(256) pack_all_kernel(const d3fk_pack_params* __restrict__ tab, int count) {
  pdl_enter();
  __shared__ float tile[PK_T][PK_MAXCOL + 1];
  __shared__ int s_layer;
  if (threadIdx.x == 0) {
    int lo = 0, hi = count - 1;                       // last entry with blk0 <= blockIdx.x
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (tab[mid].blk0 <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
    }
    s_layer = lo;
  }
  __syncthreads();
  const d3fk_pack_params p = tab[s_layer];
  const int taps = p.kh * p.kw;
  const int cib = (p.Cin + PK_T - 1) / PK_T;
  const int local = (int)blockIdx.x - p.blk0;
  const int co0 = (local / cib) * PK_T, ci0 = (local % cib) * PK_T;
  const int nco = min(PK_T, p.Cout - co0), nci = min(PK_T, p.Cin - ci0);
  const int ncol = nci * taps;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  for (int r = warp; r < nco; r += nwarp) {
    const float* src = p.w + ((long long)(co0 + r) * p.Cin + ci0) * taps;
    for (int c = lane; c < ncol; c += 32) tile[r][c] = __ldg(src + c);
  }
  __syncthreads();
  // bf16, full 8-channel groups (every layer but the 3-channel stem / head edges): one 16-byte store per (row, tap, 8 channels)
  // — the 2-byte-per-lane form below issued four times as many store instructions and ran at 1.1 TB/s.
  const bool vec8 = sizeof(T) == 2 && (nci & 7) == 0 && (nco & 7) == 0;
  if (p.w_fwd) {
    T* dst = (T*)p.w_fwd;
    if (vec8) {
      const int nv = nci >> 3;
      for (int it = threadIdx.x; it < nco * taps * nv; it += blockDim.x) {
        const int v = it % nv, q = it / nv;
        const int r = q / taps, t = q - r * taps;
        float x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = tile[r][(v * 8 + i) * taps + t];
        store_vec<T>(dst + ((long long)(co0 + r) * taps + t) * p.cin_pad + ci0 + v * 8, x);
      }
    } else {
      // one (row, tap) pair per warp iteration, lanes along the contiguous output channel: no per-element index division
      for (int q = warp; q < nco * taps; q += nwarp) {
        const int r = q / taps, t = q - r * taps;
        if (lane < nci) dst[((long long)(co0 + r) * taps + t) * p.cin_pad + ci0 + lane] = from_f<T>(tile[r][lane * taps + t]);
      }
    }
  }
  if (p.w_dgrad) {
    T* dst = (T*)p.w_dgrad;
    if (vec8) {
      const int nv = nco >> 3;
      for (int it = threadIdx.x; it < nci * taps * nv; it += blockDim.x) {
        const int v = it % nv, q = it / nv;
        const int c = q / taps, t = q - c * taps;
        float x[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = tile[v * 8 + i][c * taps + t];
        store_vec<T>(dst + ((long long)(ci0 + c) * taps + t) * p.cout_pad + co0 + v * 8, x);
      }
    } else {
      for (int q = warp; q < nci * taps; q += nwarp) {
        const int c = q / taps, t = q - c * taps;
        if (lane < nco) dst[((long long)(ci0 + c) * taps + t) * p.cout_pad + co0 + lane] = from_f<T>(tile[lane][c * taps + t]);
      }
    }
  }
}

// fused Adam (+ optional EMA lerp) over a flat arena: 16-byte accesses, streaming (28 B/param of HBM traffic)
__device__ __forceinline__ void adam_one(float& w, float g, float& m, float& v, const d3fk_adam_params& p, float step, float rsb2) {
  g *= p.grad_scale;
  m = m + (1.f - p.beta1) * (g - m);
  v = p.beta2 * v + (1.f - p.beta2) * g * g;
  const float denom = sqrtf(v) * rsb2 + p.eps;
  w = w - step * (m / denom);
}
__global__ void __launch_bounds__(256) adam_kernel(d3fk_adam_params p) {
  pdl_enter();
  if (p.dyn) {      // per-step scalars from device memory (graph replay); written by the host before the replay
    p.lr = __ldg(p.dyn); p.bias1 = __ldg(p.dyn + 1); p.bias2 = __ldg(p.dyn + 2); p.ema_decay = __ldg(p.dyn + 3);
  }
  const float step = p.lr / p.bias1;
  const float rsb2 = rsqrtf(p.bias2);
  const long long nvec = p.n >> 2;
  float4* P = reinterpret_cast<float4*>(p.p);
  const float4* G = reinterpret_cast<const float4*>(p.g);
  float4* M = reinterpret_cast<float4*>(p.m);
  float4* V = reinterpret_cast<float4*>(p.v);
  float4* E = reinterpret_cast<float4*>(p.ema);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    float4 w = P[i], m = M[i], v = V[i];
    const float4 g = __ldcs(G + i);
    adam_one(w.x, g.x, m.x, v.x, p, step, rsb2);
    adam_one(w.y, g.y, m.y, v.y, p, step, rsb2);
    adam_one(w.z, g.z, m.z, v.z, p, step, rsb2);
    adam_one(w.w, g.w, m.w, v.w, p, step, rsb2);
    M[i] = m; V[i] = v; P[i] = w;
    if (E) {
      float4 e = E[i];
      const float k = 1.f - p.ema_decay;
      e.x += k * (w.x - e.x); e.y += k * (w.y - e.y); e.z += k * (w.z - e.z); e.w += k * (w.w - e.w);
      E[i] = e;
    }
  }
  // tail (n not a multiple of 4)
  for (long long i = (nvec << 2) + blockIdx.x * (long long)blockDim.x + threadIdx.x; i < p.n; i += (long long)gridDim.x * blockDim.x) {
    float w = p.p[i], m = p.m[i], v = p.v[i];
    adam_one(w, p.g[i], m, v, p, step, rsb2);
    p.m[i] = m; p.v[i] = v; p.p[i] = w;
    if (p.ema) { float e = p.ema[i]; p.ema[i] = e + (1.f - p.ema_decay) * (w - e); }
  }
}

// ---------------------------------------------------------------------------------------------
// Video-frame pre / post-processing (d3f/train_deep_fake/lit_module.py:272-300).  HBM-bound byte shuffles: 3 B read + 12 B
// written per pixel one way, 12 B + 3 B the other.  A thread owns 4 consecutive pixels of one image: 12 contiguous frame
// bytes (three 32-bit words) on the HWC side, one float4 per colour plane on the NCHW side; H*W % 4 == 0 is required (the
// network needs H, W % 32 == 0 anyway).  BGR <-> RGB is the index 2 - c.
__global__ void __launch_bounds__(256) frames_to_tensor_kernel(d3fk_frames_params p) {
  pdl_enter();
  const long long hw = (long long)p.H * p.W, q_per_img = hw >> 2, total = q_per_img * p.N;
  float m255[3], s255[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) { m255[c] = __fmul_rn(p.mean[c], 255.f); s255[c] = __fmul_rn(p.std[c], 255.f); }
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / q_per_img, q = i - n * q_per_img;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(p.frames + (n * hw + 4 * q) * 3);
    uint32_t w[3] = {__ldcs(src), __ldcs(src + 1), __ldcs(src + 2)};
    const uint8_t* b = reinterpret_cast<const uint8_t*>(w);          // b[3*pix + {0:B, 1:G, 2:R}]
#pragma unroll
    for (int c = 0; c < 3; ++c) {                                    // c: RGB plane
      float4 o;
      o.x = __fdiv_rn(__fsub_rn((float)b[0 + 2 - c], m255[c]), s255[c]);
      o.y = __fdiv_rn(__fsub_rn((float)b[3 + 2 - c], m255[c]), s255[c]);
      o.z = __fdiv_rn(__fsub_rn((float)b[6 + 2 - c], m255[c]), s255[c]);
      o.w = __fdiv_rn(__fsub_rn((float)b[9 + 2 - c], m255[c]), s255[c]);
      reinterpret_cast<float4*>(p.tensor + (n * 3 + c) * hw)[q] = o;
    }
  }
}

__device__ __forceinline__ uint32_t denorm_u8(float t, float s255, float m255) {
  const float v = __fadd_rn(__fmul_rn(t, s255), m255);              // tensor *= std*255; tensor += mean*255 (two roundings)
  int iv = (v != v) ? 0 : (v >= 2147483648.f ? 2147483647 : (v <= -2147483648.f ? (-2147483647 - 1) : (int)v));   // .int(): toward zero
  iv = min(max(iv, 0), 255);
  return (uint32_t)iv;
}
__global__ void __launch_bounds__(256) tensor_to_frames_kernel(d3fk_frames_params p) {
  pdl_enter();
  const long long hw = (long long)p.H * p.W, q_per_img = hw >> 2, total = q_per_img * p.N;
  float m255[3], s255[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) { m255[c] = __fmul_rn(p.mean[c], 255.f); s255[c] = __fmul_rn(p.std[c], 255.f); }
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / q_per_img, q = i - n * q_per_img;
    uint32_t w[3] = {0u, 0u, 0u};
    uint8_t* b = reinterpret_cast<uint8_t*>(w);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float4 t = __ldcs(reinterpret_cast<const float4*>(p.tensor + (n * 3 + c) * hw) + q);
      b[0 + 2 - c] = (uint8_t)denorm_u8(t.x, s255[c], m255[c]);
      b[3 + 2 - c] = (uint8_t)denorm_u8(t.y, s255[c], m255[c]);
      b[6 + 2 - c] = (uint8_t)denorm_u8(t.z, s255[c], m255[c]);
      b[9 + 2 - c] = (uint8_t)denorm_u8(t.w, s255[c], m255[c]);
    }
    uint32_t* dst = reinterpret_cast<uint32_t*>(p.frames + (n * hw + 4 * q) * 3);
    dst[0] = w[0]; dst[1] = w[1]; dst[2] = w[2];
  }
}

// ---------------------------------------------------------------------------------------------
// launchers
#define DISPATCH_T(dtype, ...)                                   \
  if ((dtype) == D3FK_F32) { using T = float; __VA_ARGS__; }     \
  else if ((dtype) == D3FK_BF16) { using T = __nv_bfloat16; __VA_ARGS__; } \
  else return set_error(D3FK_ERR_ARG, "bad dtype %d", (int)(dtype));

int launch_nchw_to_nhwc(const d3fk_layout_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->cpad % 8 == 0 && p->C <= p->cpad, "cpad must be a multiple of 8 and >= C");
  D3FK_CHECK_ARG(!p->chansum || p->C <= 8, "chansum: C <= 8");
  long long total = (long long)p->B * p->H * p->W;
  DISPATCH_T(p->dtype, launch_k(nchw_to_nhwc_kernel<T>, dim3(grid_for(total, 256)), dim3(256), 0, s, dim3(1, 1, 1), p->src, (T*)p->dst, p->B, p->C, p->H * p->W, p->cpad, p->chansum));
  count_launch();
  return check_launch("nchw_to_nhwc");
}
int launch_nchw_to_s2d(const d3fk_layout_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->dtype == D3FK_BF16 && p->C == 3 && p->cpad == 4 && p->H % 2 == 0 && p->W % 2 == 0, "s2d: bf16, C = 3, cpad = 4, even H and W");
  D3FK_CHECK_ARG((((uintptr_t)p->src) & 7) == 0 && (((uintptr_t)p->dst) & 15) == 0, "s2d: alignment");
  const long long total = (long long)p->B * (p->H / 2) * (p->W / 2);
  launch_k(nchw_to_s2d_kernel, dim3(grid_for(total, 256)), dim3(256), 0, s, dim3(1, 1, 1), p->src, (__nv_bfloat16*)p->dst, p->B, p->H, p->W);
  count_launch();
  return check_launch("nchw_to_s2d");
}
int launch_pack_stem(const d3fk_pack_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->dtype == D3FK_BF16 && p->Cin == 3 && p->kh == 7 && p->kw == 7 && p->w && p->w_fwd, "pack_stem: bf16 7x7 stem weights");
  launch_k(pack_stem_kernel, dim3(cdiv(p->Cout * 256, 256)), dim3(256), 0, s, dim3(1, 1, 1), p->w, (__nv_bfloat16*)p->w_fwd, p->Cout);
  count_launch();
  return check_launch("pack_stem");
}
int launch_bn_finalize(const d3fk_bn_params* p, cudaStream_t s) {
  launch_k(bn_finalize_kernel, dim3(cdiv(p->C, 128)), dim3(128), 0, s, dim3(1, 1, 1), *p);
  count_launch();
  return check_launch("bn_finalize");
}
int launch_bn_fold(const d3fk_bn_params* p, cudaStream_t s) {
  launch_k(bn_fold_kernel, dim3(cdiv(p->C, 128)), dim3(128), 0, s, dim3(1, 1, 1), *p);
  count_launch();
  return check_launch("bn_fold");
}
int launch_bn_apply(const d3fk_bn_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->C % 8 == 0, "C must be a multiple of 8");
  int V = p->dtype == D3FK_F32 ? 4 : 8;
  long long total = p->count * (p->C / V);
  D3FK_CHECK_ARG(256 % (p->C / V) == 0, "C / vector width must divide 256 (the kernel's channel vector is loop invariant)");
  DISPATCH_T(p->dtype, launch_k(bn_apply_kernel<T>, dim3(grid_for(total, 256 * 4, D3FK_BN_BWD_BLOCKS)), dim3(256), 2 * p->C * sizeof(float), s, dim3(1, 1, 1), *p));
  count_launch();
  return check_launch("bn_apply");
}
int launch_bn_bwd_reduce(const d3fk_bn_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->C % 8 == 0 && p->C <= 1024, "C must be a multiple of 8, <= 1024");
  int V = p->dtype == D3FK_F32 ? 4 : 8;
  int cvs = p->C / V;
  D3FK_CHECK_ARG((cvs & (cvs - 1)) == 0 && cvs <= 256, "C/V must be a power of two <= 256");
  const int threads = 256;
  const int rows = threads / cvs;
  int grid = cdiv(p->count, (long long)rows * 8);
  if (grid > kSMs * 8) grid = kSMs * 8;
  if (grid < 1) grid = 1;
  const int slotC = cvs < 32 ? p->C : 32 * V;
  size_t smem = (size_t)(threads / 32) * 2 * slotC * sizeof(double);
  const bool xm = p->relu && p->mask_from_x;
  D3FK_CHECK_ARG(!xm || (p->scale && p->shift), "mask_from_x needs scale / shift");
  if (p->dtype == D3FK_F32) {
    if (xm) launch_k(bn_bwd_reduce_kernel<float, double, true>, dim3(grid), dim3(threads), smem, s, dim3(1, 1, 1), *p);
    else launch_k(bn_bwd_reduce_kernel<float, double, false>, dim3(grid), dim3(threads), smem, s, dim3(1, 1, 1), *p);
  } else if (p->dtype == D3FK_BF16) {
    if (xm) launch_k(bn_bwd_reduce_kernel<__nv_bfloat16, float, true>, dim3(grid), dim3(threads), smem, s, dim3(1, 1, 1), *p);
    else launch_k(bn_bwd_reduce_kernel<__nv_bfloat16, float, false>, dim3(grid), dim3(threads), smem, s, dim3(1, 1, 1), *p);
  } else return set_error(D3FK_ERR_ARG, "bad dtype");
  count_launch();
  return check_launch("bn_bwd_reduce");
}
int launch_bn_bwd_finalize(const d3fk_bn_params* p, cudaStream_t s) {
  launch_k(bn_bwd_finalize_kernel, dim3(cdiv(p->C, 128)), dim3(128), 0, s, dim3(1, 1, 1), *p);
  count_launch();
  return check_launch("bn_bwd_finalize");
}
int launch_bn_bwd_apply(const d3fk_bn_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->C % 8 == 0, "C must be a multiple of 8");
  int V = p->dtype == D3FK_F32 ? 4 : 8;
  long long total = p->count * (p->C / V);
  D3FK_CHECK_ARG(256 % (p->C / V) == 0, "C / vector width must divide 256 (the kernel's channel vector is loop invariant)");
  const bool xm = p->relu && p->mask_from_x;
  D3FK_CHECK_ARG(!xm || (p->scale && p->shift), "mask_from_x needs scale / shift");
  if (xm) { DISPATCH_T(p->dtype, launch_k(bn_bwd_apply_kernel<T, true>, dim3(grid_for(total, 256 * 4, D3FK_BN_BWD_BLOCKS)), dim3(256), 6 * p->C * sizeof(float), s, dim3(1, 1, 1), *p)); }
  else { DISPATCH_T(p->dtype, launch_k(bn_bwd_apply_kernel<T, false>, dim3(grid_for(total, 256 * 4, D3FK_BN_BWD_BLOCKS)), dim3(256), 6 * p->C * sizeof(float), s, dim3(1, 1, 1), *p)); }
  count_launch();
  return check_launch("bn_bwd_apply");
}
static int launch_bn_bwd_frozen(const d3fk_bn_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->C % 8 == 0 && p->C <= 1024, "C must be a multiple of 8, <= 1024");
  D3FK_CHECK_ARG(p->dx && p->bstats && p->gamma && p->invstd && p->mean, "frozen BN backward: dx, bstats, gamma, mean, invstd");
  const int V = p->dtype == D3FK_F32 ? 4 : 8;
  const int cvs = p->C / V;
  D3FK_CHECK_ARG((cvs & (cvs - 1)) == 0 && cvs <= 256, "C/V must be a power of two <= 256");
  const int threads = 256;
  const int rows = threads / cvs;
  int grid = cdiv(p->count, (long long)rows * 8);
  if (grid > kSMs * 8) grid = kSMs * 8;
  if (grid < 1) grid = 1;
  const int slotC = cvs < 32 ? p->C : 32 * V;
  size_t smem = (size_t)(threads / 32) * 2 * slotC * sizeof(double);
  if (smem < 3 * (size_t)p->C * sizeof(float)) smem = 3 * (size_t)p->C * sizeof(float);
  const bool xm = p->relu && p->mask_from_x;
  D3FK_CHECK_ARG(!xm || (p->scale && p->shift), "mask_from_x needs scale / shift");
  if (p->dtype == D3FK_F32) {
    if (xm) launch_k(bn_bwd_frozen_kernel<float, double, true>, dim3(grid), dim3(threads), smem, s, dim3(1, 1, 1), *p);
    else launch_k(bn_bwd_frozen_kernel<float, double, false>, dim3(grid), dim3(threads), smem, s, dim3(1, 1, 1), *p);
  } else if (p->dtype == D3FK_BF16) {
    if (xm) launch_k(bn_bwd_frozen_kernel<__nv_bfloat16, float, true>, dim3(grid), dim3(threads), smem, s, dim3(1, 1, 1), *p);
    else launch_k(bn_bwd_frozen_kernel<__nv_bfloat16, float, false>, dim3(grid), dim3(threads), smem, s, dim3(1, 1, 1), *p);
  } else return set_error(D3FK_ERR_ARG, "bad dtype");
  count_launch();
  int rc = check_launch("bn_bwd_frozen");
  return rc ? rc : launch_bn_bwd_finalize(p, s);
}
int launch_bn_bwd(const d3fk_bn_params* p, cudaStream_t s) {
  if (p->frozen) return launch_bn_bwd_frozen(p, s);
  D3FK_CHECK_ARG(p->C % 8 == 0 && p->C <= 1024, "C must be a multiple of 8, <= 1024");
  const int V = p->dtype == D3FK_F32 ? 4 : 8;
  const int cvs = p->C / V;
  const bool pow2 = (cvs & (cvs - 1)) == 0 && cvs <= 256;
  // one launch only where latency dominates (tensor <= 4 M elements: L2-resident second pass); big layers stream twice
  if (!p->barrier || !pow2 || !g_fuse_bn_bwd || p->count * (long long)p->C > g_fuse_bn_bwd_max) {
    int rc = launch_bn_bwd_reduce(p, s);
    return rc ? rc : launch_bn_bwd_apply(p, s);
  }
  const int threads = 256;
  const int rows = threads / cvs;
  // co-resident grid: at most 2 blocks per SM (launch bounds), sized like the reduce kernel
  int grid = cdiv(p->count, (long long)rows * 8);
  if (grid > kSMs * 2) grid = kSMs * 2;
  if (grid < 1) grid = 1;
  const int slotC = cvs < 32 ? p->C : 32 * V;
  size_t smem = (size_t)(threads / 32) * 2 * slotC * sizeof(double);
  const size_t smem_apply = 6 * (size_t)p->C * sizeof(float);
  if (smem_apply > smem) smem = smem_apply;
  const bool xm = p->relu && p->mask_from_x;
  D3FK_CHECK_ARG(!xm || (p->scale && p->shift), "mask_from_x needs scale / shift");
  if (p->dtype == D3FK_F32) {
    if (xm) launch_k(bn_bwd_kernel<float, double, true>, dim3(grid), dim3(threads), smem, s, dim3(1, 1, 1), *p, g_dev_error_flag);
    else launch_k(bn_bwd_kernel<float, double, false>, dim3(grid), dim3(threads), smem, s, dim3(1, 1, 1), *p, g_dev_error_flag);
  } else if (p->dtype == D3FK_BF16) {
    if (xm) launch_k(bn_bwd_kernel<__nv_bfloat16, float, true>, dim3(grid), dim3(threads), smem, s, dim3(1, 1, 1), *p, g_dev_error_flag);
    else launch_k(bn_bwd_kernel<__nv_bfloat16, float, false>, dim3(grid), dim3(threads), smem, s, dim3(1, 1, 1), *p, g_dev_error_flag);
  } else return set_error(D3FK_ERR_ARG, "bad dtype");
  count_launch();
  return check_launch("bn_bwd");
}
int launch_maxpool_fwd(const d3fk_pool_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->C % 8 == 0 && p->H % 2 == 0 && p->W % 2 == 0, "C%8, H%2, W%2");
  int V = p->dtype == D3FK_F32 ? 4 : 8;
  long long total = (long long)p->B * (p->H / 2) * (p->W / 2) * (p->C / V);
  DISPATCH_T(p->dtype, launch_k(maxpool_fwd_kernel<T>, dim3(grid_for(total, 256)), dim3(256), 0, s, dim3(1, 1, 1), *p));
  count_launch();
  return check_launch("maxpool_fwd");
}
int launch_maxpool_bwd(const d3fk_pool_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->C % 8 == 0 && p->idx && p->H % 2 == 0 && p->W % 2 == 0, "C%8, H%2, W%2 and idx required");
  int V = p->dtype == D3FK_F32 ? 4 : 8;
  long long total = (long long)p->B * (p->H / 2) * (p->W / 2) * (p->C / V);      // one thread per 2x2 block of dx and channel vector
  DISPATCH_T(p->dtype, launch_k(maxpool_bwd_kernel<T>, dim3(grid_for(total, 256)), dim3(256), 0, s, dim3(1, 1, 1), *p));
  count_launch();
  return check_launch("maxpool_bwd");
}
int launch_sumpool2(const d3fk_pool_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->C % 8 == 0, "C%8");
  int V = p->dtype == D3FK_F32 ? 4 : 8;
  long long total = (long long)p->B * p->H * p->W * (p->C / V);
  DISPATCH_T(p->dtype, launch_k(sumpool2_kernel<T>, dim3(grid_for(total, 256)), dim3(256), 0, s, dim3(1, 1, 1), *p));
  count_launch();
  return check_launch("sumpool2");
}
int launch_upcat(const d3fk_upcat_params* p, cudaStream_t s) {
  int V = p->dtype == D3FK_F32 ? 4 : 8;
  D3FK_CHECK_ARG(p->c0 % V == 0 && p->c1 % V == 0 && p->ld0 % V == 0 && p->ldo % V == 0 && (p->c1 == 0 || p->ld1 % V == 0),
                 "channel counts and pixel strides must be multiples of the 16-byte vector");
  D3FK_CHECK_ARG(p->H % 2 == 0 && p->W % 2 == 0 && p->c0 > 0, "H, W even, c0 > 0");
  long long rows = (long long)p->B * p->H;
  const unsigned grid = (unsigned)(rows < (1ll << 30) ? rows : (1ll << 30));
  DISPATCH_T(p->dtype, launch_k(upcat_kernel<T>, dim3(grid), dim3(256), 0, s, dim3(1, 1, 1), *p));
  count_launch();
  return check_launch("upcat");
}
int launch_chansum(const d3fk_chansum_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->C <= 8 && p->ld % 8 == 0, "C<=8, ld%8");
  DISPATCH_T(p->dtype, launch_k(chansum_kernel<T>, dim3(grid_for(p->count, 256, 2)), dim3(256), 0, s, dim3(1, 1, 1), *p));
  count_launch();
  return check_launch("chansum");
}
int launch_qsample(const d3fk_qsample_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->chw % 4 == 0, "C*H*W must be a multiple of 4");
  D3FK_CHECK_ARG(p->B >= 1 && p->B <= 65535, "batch must be 1..65535");
  const int vps = p->chw / 4;
  int gx = cdiv(vps, 256 * 4);                    // ~4 vectors per thread; enough blocks per sample to fill the chip at small B
  const int want = cdiv(148 * 8, p->B);
  if (gx < want) gx = want < cdiv(vps, 256) ? want : cdiv(vps, 256);
  if (gx < 1) gx = 1;
  launch_k(qsample_kernel, dim3(gx, p->B), dim3(256), 0, s, dim3(1, 1, 1), *p);
  count_launch();
  return check_launch("q_sample");
}
int launch_affine_qsample(const d3fk_affine_qsample_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->B >= 1 && p->B <= 65535 && p->C >= 1 && p->H >= 1, "batch must be 1..65535, C and H positive");
  D3FK_CHECK_ARG(p->W >= 4 && p->W % 4 == 0, "W must be a multiple of 4");
  D3FK_CHECK_ARG(p->x && p->minv && p->out_noisy, "x, minv and out_noisy are required");
  D3FK_CHECK_ARG((long long)p->C * p->H * p->W < (1ll << 31), "one sample must have fewer than 2^31 elements");
  const int vps = p->C * p->H * p->W / 4;
  int gx = cdiv(vps, 256 * 2);
  const int want = cdiv(148 * 8, p->B);
  if (gx < want) gx = want < cdiv(vps, 256) ? want : cdiv(vps, 256);
  if (gx < 1) gx = 1;
  launch_k(affine_qsample_kernel, dim3(gx, p->B), dim3(256), 0, s, dim3(1, 1, 1), *p);
  count_launch();
  return check_launch("affine_q_sample");
}
int launch_posterior(const d3fk_posterior_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->n % 4 == 0, "n must be a multiple of 4");
  if (!p->mask) {
    launch_k(posterior_kernel, dim3(grid_for(p->n / 4, 256)), dim3(256), 0, s, dim3(1, 1, 1), *p);
    count_launch();
    return check_launch("posterior_step");
  }
  D3FK_CHECK_ARG(p->src && p->x && p->x0_hat, "the masked posterior needs x, x0_hat and src");
  D3FK_CHECK_ARG(p->hw > 0 && p->hw % 4 == 0 && p->chw >= p->hw && p->chw % p->hw == 0, "hw must be a multiple of 4 dividing chw");
  D3FK_CHECK_ARG(p->n > 0 && p->n % p->chw == 0 && p->n / p->chw <= 65535, "n must be 1..65535 samples of chw elements");
  D3FK_CHECK_ARG((((uintptr_t)p->x | (uintptr_t)p->x0_hat | (uintptr_t)p->src | (uintptr_t)p->mask | (uintptr_t)p->z |
                   (uintptr_t)p->known_noise) & 15) == 0, "buffers must be 16-byte aligned");
  const int gx = cdiv(p->chw / 4, 256);           // one 4-element vector per thread
  launch_k(posterior_masked_kernel, dim3(gx, (unsigned)(p->n / p->chw)), dim3(256), 0, s, dim3(1, 1, 1), *p);
  count_launch();
  return check_launch("posterior_step");
}
static bool overlaps(const void* a, const void* b, long long bytes) {
  return a && b && (uintptr_t)a < (uintptr_t)b + bytes && (uintptr_t)b < (uintptr_t)a + bytes;
}
int launch_posterior_2m(const d3fk_posterior_2m_params* p, cudaStream_t s) {
  const d3fk_posterior_params* q = &p->base;
  D3FK_CHECK_ARG(q->n % 4 == 0, "n must be a multiple of 4");
  D3FK_CHECK_ARG(q->x && q->x0_hat && p->x0_prev, "the 2M posterior needs x, x0_hat and x0_prev");
  D3FK_CHECK_ARG(!overlaps(p->x0_prev, q->x0_hat, q->n * 4) && !overlaps(p->x0_prev, q->x, q->n * 4),
                 "x0_prev must not overlap x0_hat or x");
  D3FK_CHECK_ARG(((uintptr_t)p->x0_prev & 15) == 0, "x0_prev must be 16-byte aligned");
  if (!q->mask) {
    launch_k(posterior_2m_kernel, dim3(grid_for(q->n / 4, 256)), dim3(256), 0, s, dim3(1, 1, 1), *p);
    count_launch();
    return check_launch("posterior_2m_step");
  }
  D3FK_CHECK_ARG(q->src, "the masked posterior needs src");
  D3FK_CHECK_ARG(q->hw > 0 && q->hw % 4 == 0 && q->chw >= q->hw && q->chw % q->hw == 0, "hw must be a multiple of 4 dividing chw");
  D3FK_CHECK_ARG(q->n > 0 && q->n % q->chw == 0 && q->n / q->chw <= 65535, "n must be 1..65535 samples of chw elements");
  D3FK_CHECK_ARG((((uintptr_t)q->x | (uintptr_t)q->x0_hat | (uintptr_t)q->src | (uintptr_t)q->mask | (uintptr_t)q->z |
                   (uintptr_t)q->known_noise) & 15) == 0, "buffers must be 16-byte aligned");
  const int gx = cdiv(q->chw / 4, 256);
  launch_k(posterior_2m_masked_kernel, dim3(gx, (unsigned)(q->n / q->chw)), dim3(256), 0, s, dim3(1, 1, 1), *p);
  count_launch();
  return check_launch("posterior_2m_step");
}
int launch_inc(const d3fk_misc_params* p, cudaStream_t s) {
  launch_k(inc_kernel, dim3(1), dim3(1), 0, s, dim3(1, 1, 1), (int*)p->p0);
  count_launch();
  return check_launch("inc");
}
int launch_pack_all(const d3fk_misc_params* p, cudaStream_t s) {
  // p0: device array of d3fk_pack_params (same dtype, blk0 = running block count, every layer with taps * min(Cin,32)
  // <= 288); n = (total blocks << 17) | (count << 1) | (dtype == bf16)
  const int count = (int)((p->n >> 1) & 0xFFFF);
  const long long blocks = p->n >> 17;
  D3FK_CHECK_ARG(count > 0 && blocks > 0 && blocks < (1ll << 31), "bad pack table");
  if (p->n & 1) launch_k(pack_all_kernel<__nv_bfloat16>, dim3((unsigned)blocks), dim3(256), 0, s, dim3(1, 1, 1), (const d3fk_pack_params*)p->p0, count);
  else launch_k(pack_all_kernel<float>, dim3((unsigned)blocks), dim3(256), 0, s, dim3(1, 1, 1), (const d3fk_pack_params*)p->p0, count);
  count_launch();
  return check_launch("pack_all");
}
static int check_frames(const d3fk_frames_params* p) {
  D3FK_CHECK_ARG(p->N > 0 && p->H > 0 && p->W > 0 && p->frames && p->tensor, "empty batch or null buffer");
  D3FK_CHECK_ARG(((long long)p->H * p->W) % 4 == 0, "H*W must be a multiple of 4");
  D3FK_CHECK_ARG((((uintptr_t)p->frames) & 3) == 0 && (((uintptr_t)p->tensor) & 15) == 0, "frames must be 4-byte and tensor 16-byte aligned");
  D3FK_CHECK_ARG(p->std[0] != 0.f && p->std[1] != 0.f && p->std[2] != 0.f, "std must be non-zero");
  return D3FK_OK;
}
int launch_frames_to_tensor(const d3fk_frames_params* p, cudaStream_t s) {
  int rc = check_frames(p);
  if (rc) return rc;
  launch_k(frames_to_tensor_kernel, dim3(grid_for((long long)p->N * p->H * p->W / 4, 256)), dim3(256), 0, s, dim3(1, 1, 1), *p);
  count_launch();
  return check_launch("frames_to_tensor");
}
int launch_tensor_to_frames(const d3fk_frames_params* p, cudaStream_t s) {
  int rc = check_frames(p);
  if (rc) return rc;
  launch_k(tensor_to_frames_kernel, dim3(grid_for((long long)p->N * p->H * p->W / 4, 256)), dim3(256), 0, s, dim3(1, 1, 1), *p);
  count_launch();
  return check_launch("tensor_to_frames");
}
__global__ void set_scalars_kernel(d3fk_scalars_params p) {
  pdl_enter();
  if (threadIdx.x < 4) p.dst[threadIdx.x] = p.v[threadIdx.x];
}
int launch_set_scalars(const d3fk_scalars_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->dst != nullptr, "dst is null");
  launch_k(set_scalars_kernel, dim3(1), dim3(32), 0, s, dim3(1, 1, 1), *p);
  count_launch();
  return check_launch("set_scalars");
}

int launch_adam(const d3fk_adam_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG((((uintptr_t)p->p | (uintptr_t)p->g | (uintptr_t)p->m | (uintptr_t)p->v | (uintptr_t)p->ema) & 15) == 0, "arenas must be 16-byte aligned");
  launch_k(adam_kernel, dim3(grid_for(p->n / 4 + 1, 256)), dim3(256), 0, s, dim3(1, 1, 1), *p);
  count_launch();
  return check_launch("adam");
}

}  // namespace d3fk
