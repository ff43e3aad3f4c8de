// loss.cu — fused MSE + (1 - SSIM) criterion, forward AND gradient in one kernel.
// Reference: d3f/loss_functions/structural_similarity_loss.py:14-26 with piqa.SSIM() defaults (11-tap Gaussian,
// sigma 1.5, valid window, k1 = 0.01, k2 = 0.03, value_range 1; SURVEY Appendix B1).  ~30 eager launches -> 1.
//
// One block owns a 32x32 pixel tile of one (n, c) plane.  It stages the clipped, normalised inputs with a 10-pixel
// halo (52x52), runs the separable Gaussian over {x, y, x^2, y^2, xy} for the 42x42 windows that touch the tile,
// forms ss and its partials a = d ss/d mu_x, b = d ss/d E[x^2], c = d ss/d E[xy], pushes them back through the
// transposed separable filter and emits dL/dpred for its 32x32 pixels.  Everything between load and store lives in
// shared memory; HBM traffic is one read of pred/target and one write of the gradient.
#include "common.cuh"

namespace d3fk {

constexpr int LT = 32;            // tile edge
constexpr int LW = 11;            // window
constexpr int LH = LW - 1;        // halo
constexpr int LI = LT + 2 * LH;   // 52: staged input edge
constexpr int LM = LT + LH;       // 42: windows (map pixels) touching the tile
// the a / b / c maps reuse the staged-input region (dead after the horizontal pass; 3*42*42 <= 2*52*52): 65 KB per block,
// three blocks per SM instead of two
constexpr int LOSS_SMEM = (2 * LI * LI + 5 * LI * LM) * 4;
static_assert(3 * LM * LM <= 2 * LI * LI, "the derivative maps must fit the staged-input region");

__global__ void __launch_bounds__(256, 3) mse_ssim_loss_kernel(d3fk_loss_params p) {
  pdl_enter();
  extern __shared__ float sm[];
  float* xs = sm;                       // [LI][LI] normalised clipped prediction (0 outside the image)
  float* ys = xs + LI * LI;             // [LI][LI] target
  float* hs = ys + LI * LI;             // [5][LI][LM] horizontal pass; later [3][LM][LT] transposed horizontal pass
  float* ms = xs;                       // [3][LM][LM] a, b, c maps — over xs / ys, which are dead once step 2 is done
  __shared__ float g[LW];
  __shared__ double red[2][8];
  const int tid = threadIdx.x;
  if (tid < LW) g[tid] = p.win[tid];
  const int tiles_w = p.W / LT, tiles_h = p.H / LT;
  int b = blockIdx.x;
  const int tw = b % tiles_w; b /= tiles_w;
  const int th = b % tiles_h; b /= tiles_h;
  const long long plane = (long long)b * p.H * p.W;     // b = n*C + c
  const int r0 = th * LT - LH, c0 = tw * LT - LH;       // image coords of staged (0,0)
  const float inv_range = 1.0f / (p.hi - p.lo);
  const int Hm = p.H - LH, Wm = p.W - LH;               // valid window (map) extent

  // 1. stage inputs.  All of a thread's 2 x 11 global loads are issued before the first one is used: as a plain loop
  //    (load, transform, store per element) this phase exposed the HBM latency ~11 times per block and held 27 % of the
  //    kernel's stall samples (ncu, r01g).
  {
    constexpr int NST = (LI * LI + 255) / 256;
    float px[NST], py[NST];
#pragma unroll
    for (int k = 0; k < NST; ++k) {
      const int i = tid + 256 * k;
      const int r = i / LI, c = i - r * LI;
      const int gr = r0 + r, gc = c0 + c;
      const bool ok = i < LI * LI && (unsigned)gr < (unsigned)p.H && (unsigned)gc < (unsigned)p.W;
      const long long o = ok ? plane + (long long)gr * p.W + gc : plane;
      px[k] = ok ? __ldg(p.pred + o) : p.lo;          // lo normalises to 0: the value staged outside the image
      py[k] = ok ? __ldg(p.target + o) : p.lo;
    }
#pragma unroll
    for (int k = 0; k < NST; ++k) {
      const int i = tid + 256 * k;
      if (i < LI * LI) {
        xs[i] = fminf(fmaxf((px[k] - p.lo) * inv_range, 0.f), 1.f);
        ys[i] = fminf(fmaxf((py[k] - p.lo) * inv_range, 0.f), 1.f);
      }
    }
  }
  __syncthreads();
  // 2. horizontal Gaussian of x, y, xx, yy, xy : hs[q][r][jc], window columns jc..jc+10.
  //    Register blocking: a thread produces 3 adjacent outputs from 13 staged inputs (the passes are LDS-bound).
  for (int i = tid; i < LI * (LM / 3); i += 256) {
    const int r = i / (LM / 3), jc = (i - r * (LM / 3)) * 3;
    float xv[LW + 2], yv[LW + 2];
#pragma unroll
    for (int k = 0; k < LW + 2; ++k) { xv[k] = xs[r * LI + jc + k]; yv[k] = ys[r * LI + jc + k]; }
#pragma unroll
    for (int o = 0; o < 3; ++o) {
      float sx = 0.f, sy = 0.f, sxx = 0.f, syy = 0.f, sxy = 0.f;
#pragma unroll
      for (int k = 0; k < LW; ++k) {
        const float x = xv[o + k], y = yv[o + k], w = g[k];
        sx = fmaf(w, x, sx); sy = fmaf(w, y, sy);
        sxx = fmaf(w, x * x, sxx); syy = fmaf(w, y * y, syy); sxy = fmaf(w, x * y, sxy);
      }
      const int idx = r * LM + jc + o;
      hs[0 * LI * LM + idx] = sx; hs[1 * LI * LM + idx] = sy; hs[2 * LI * LM + idx] = sxx;
      hs[3 * LI * LM + idx] = syy; hs[4 * LI * LM + idx] = sxy;
    }
  }
  __syncthreads();
  // 3. vertical Gaussian -> ss and its partial derivatives at every window that touches the tile
  //    (3 vertically adjacent windows per thread: 13 rows of each map feed 3 x 11 taps)
  const float C1 = 0.01f * 0.01f, C2 = 0.03f * 0.03f;
  double ss_sum = 0.0;
  for (int i = tid; i < (LM / 3) * LM; i += 256) {
    const int jg = i / LM, jc = i - jg * LM;
    const int jr0 = jg * 3;
    float acc5[3][5];
#pragma unroll
    for (int o = 0; o < 3; ++o)
#pragma unroll
      for (int q = 0; q < 5; ++q) acc5[o][q] = 0.f;
#pragma unroll
    for (int k = 0; k < LW + 2; ++k) {
      const int o2 = (jr0 + k) * LM + jc;
      float v[5];
#pragma unroll
      for (int q = 0; q < 5; ++q) v[q] = hs[q * LI * LM + o2];
#pragma unroll
      for (int o = 0; o < 3; ++o) {
        const int kk = k - o;
        if (kk >= 0 && kk < LW) {
          const float w = g[kk];
#pragma unroll
          for (int q = 0; q < 5; ++q) acc5[o][q] = fmaf(w, v[q], acc5[o][q]);
        }
      }
    }
#pragma unroll
    for (int o = 0; o < 3; ++o) {
      const int jr = jr0 + o;
      const int gr = r0 + jr, gc = c0 + jc;                // window origin in the image
      float a = 0.f, bb = 0.f, cc = 0.f;
      if ((unsigned)gr < (unsigned)Hm && (unsigned)gc < (unsigned)Wm) {
        const float mx = acc5[o][0], my = acc5[o][1], exx = acc5[o][2], eyy = acc5[o][3], exy = acc5[o][4];
        const float mxx = mx * mx, myy = my * my, mxy = mx * my;
        const float sxx = exx - mxx, syy = eyy - myy, sxy = exy - mxy;
        const float A1 = 2.f * mxy + C1, A2 = 2.f * sxy + C2, B1 = mxx + myy + C1, B2 = sxx + syy + C2;
        const float rB1 = 1.f / B1, rB2 = 1.f / B2;          // two divisions per window instead of six
        const float S1 = A1 * rB1, S2 = A2 * rB2;
        // windows whose origin lies inside the tile are owned (counted) by this block
        if (jr >= LH && jc >= LH) ss_sum += (double)(S1 * S2);
        a = S2 * 2.f * (my - S1 * mx) * rB1 + S1 * 2.f * (S2 * mx - my) * rB2;
        bb = -S1 * S2 * rB2;
        cc = 2.f * S1 * rB2;
      }
      const int idx = jr * LM + jc;
      ms[idx] = a; ms[LM * LM + idx] = bb; ms[2 * LM * LM + idx] = cc;
    }
  }
  __syncthreads();
  double mse_sum = 0.0;
  if (p.grad) {
    // 4. transposed horizontal pass: th[q][jr][ic] = sum_{jc = ic..ic+10} g[ic+10-jc] * map[q][jr][jc]; 4 outputs / thread
    float* ths = hs;
    for (int i = tid; i < 3 * LM * (LT / 4); i += 256) {
      const int q = i / (LM * (LT / 4));
      const int rem = i - q * LM * (LT / 4);
      const int jr = rem / (LT / 4), ic = (rem - jr * (LT / 4)) * 4;
      float v[LW + 3];
#pragma unroll
      for (int k = 0; k < LW + 3; ++k) v[k] = ms[q * LM * LM + jr * LM + ic + k];
#pragma unroll
      for (int o = 0; o < 4; ++o) {
        float sacc = 0.f;
#pragma unroll
        for (int k = 0; k < LW; ++k) sacc = fmaf(g[LH - k], v[o + k], sacc);
        ths[q * LM * LT + jr * LT + ic + o] = sacc;
      }
    }
    __syncthreads();
  }
  // 5. transposed vertical pass + combination + MSE term; 4 vertically adjacent pixels per thread
  const long long ntot = (long long)p.B * p.C * p.H * p.W;
  const double nmap = (double)p.B * p.C * (double)Hm * Wm;
  const float k_mse = p.grad_scale * 0.5f * 2.0f / (float)ntot;
  const float k_ssim = p.grad_scale * 0.5f * inv_range / (float)nmap;
  for (int i = tid; i < (LT / 4) * LT; i += 256) {
    const int ig = i / LT, ic = i - ig * LT;
    const int ir0 = ig * 4;
    float A[4], Bm[4], Cm[4];
#pragma unroll
    for (int o = 0; o < 4; ++o) { A[o] = 0.f; Bm[o] = 0.f; Cm[o] = 0.f; }
    if (p.grad) {
      const float* ths = hs;
#pragma unroll
      for (int k = 0; k < LW + 3; ++k) {
        const int o2 = (ir0 + k) * LT + ic;
        const float va = ths[o2], vb = ths[LM * LT + o2], vc = ths[2 * LM * LT + o2];
#pragma unroll
        for (int o = 0; o < 4; ++o) {
          const int kk = k - o;
          if (kk >= 0 && kk < LW) {
            const float w = g[LH - kk];
            A[o] = fmaf(w, va, A[o]); Bm[o] = fmaf(w, vb, Bm[o]); Cm[o] = fmaf(w, vc, Cm[o]);
          }
        }
      }
    }
#pragma unroll
    for (int o = 0; o < 4; ++o) {
      const int ir = ir0 + o;
      const long long oidx = plane + (long long)(th * LT + ir) * p.W + tw * LT + ic;
      const float pr = __ldg(p.pred + oidx), tg = __ldg(p.target + oidx);
      const float d = pr - tg;
      mse_sum += (double)d * d;
      if (p.grad) {
        const float xn = (pr - p.lo) * inv_range;
        const float x = fminf(fmaxf(xn, 0.f), 1.f), y = fminf(fmaxf((tg - p.lo) * inv_range, 0.f), 1.f);   // as staged in step 1
        // torch's clip subgradient: 1 on the closed range [lo, hi] (a prediction exactly at lo or hi keeps its SSIM term),
        // 0 strictly outside it
        const float inside = (xn >= 0.f && xn <= 1.f) ? 1.f : 0.f;
        const float dss = A[o] + 2.f * x * Bm[o] + y * Cm[o];
        p.grad[oidx] = k_mse * d - k_ssim * inside * dss;
      }
    }
  }
  // block reduction of the two sums
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mse_sum += __shfl_xor_sync(0xffffffffu, mse_sum, o);
    ss_sum += __shfl_xor_sync(0xffffffffu, ss_sum, o);
  }
  if ((tid & 31) == 0) { red[0][tid >> 5] = mse_sum; red[1][tid >> 5] = ss_sum; }
  __syncthreads();
  if (tid < 2) {
    double a = 0;
    for (int w = 0; w < 8; ++w) a += red[tid][w];
    atomicAdd(&p.acc[tid], a);
    if (p.loss_out) __threadfence();      // only the two publishing threads fence (a block-wide fence was 3 % of the kernel)
  }
  if (p.loss_out) {
    // The last block to finish forms the scalar loss and resets the accumulators (acc[2] doubles as the ticket), so the
    // criterion is ONE launch: no memset before, no scalar arithmetic kernels after.
    __shared__ unsigned s_ticket;
    __syncthreads();
    unsigned* ticket = reinterpret_cast<unsigned*>(p.acc + 2);
    if (tid == 0) s_ticket = atomicAdd(ticket, 1u);
    __syncthreads();
    if (s_ticket == gridDim.x - 1 && tid == 0) {
      __threadfence();
      const double mse = atomicAdd(&p.acc[0], 0.0), ssum = atomicAdd(&p.acc[1], 0.0);
      *p.loss_out = (float)((mse / (double)ntot + 1.0 - ssum / nmap) * 0.5);
      p.acc[0] = 0.0; p.acc[1] = 0.0;
      *ticket = 0u;
    }
  }
}

int loss_init() {
  cudaError_t e = cudaFuncSetAttribute(mse_ssim_loss_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LOSS_SMEM);
  if (e != cudaSuccess) return set_error(D3FK_ERR_CUDA, "loss smem attribute: %s", cudaGetErrorString(e));
  return D3FK_OK;
}

int launch_loss(const d3fk_loss_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->H % LT == 0 && p->W % LT == 0, "H and W must be multiples of 32");
  D3FK_CHECK_ARG(p->hi > p->lo, "bad value range");
  long long blocks = (long long)p->B * p->C * (p->H / LT) * (p->W / LT);
  D3FK_CHECK_ARG(blocks < (1ll << 31), "too many tiles");
  launch_k(mse_ssim_loss_kernel, dim3((int)blocks), dim3(256), LOSS_SMEM, s, dim3(1, 1, 1), *p);
  count_launch();
  return check_launch("mse_ssim_loss");
}

}  // namespace d3fk
