// stem_dgrad.cu — the input gradient of the 7x7 / stride-2 / pad-3 stem convolution: dX[b][ci][h][w] (fp32 NCHW, ci < 3) from
// the stem's pre-BN gradient dY [B][H/2][W/2][64] (bf16 NHWC) and the dgrad-packed weights w[ci][kh][kw][64].
//
// Why not the generic conv mode 1: its transposed gather runs K = 49 * 64 of which ~3/4 of the taps are structurally zero (only
// kh = h + 3 (mod 2) and kw = w + 3 (mod 2) land on a dY pixel), and N = 3 pads to a 16-wide UMMA.  Here every output pixel
// belongs to one of four parity classes (h % 2, w % 2); a class sees 3 (even) or 4 (odd) taps per axis, so the classes are
// 3x3, 3x4, 4x3 and 4x4 taps (12.25 on average instead of 49), and within a class 16 consecutive pixels of a row (w, w+2, ...)
// read 16 CONSECUTIVE dY pixels for every tap.  That is a warp-level mma.sync.m16n8k16 problem (M = 16 pixels, N = 8 with 3
// real, K = 64 channels per tap in four 16-channel k-steps) fed by ldmatrix from a halo tile of dY in shared memory, like the
// head convolution's mma form (head_conv.cu).
//
// A 256-thread block owns a 32 x 32 output tile: 4 classes x 16 rows x 16 columns.  Its dY halo is 19 x 19 pixels (rows / columns
// h0/2 - 1 .. h0/2 + 17), staged as 8 channel planes of 16 bytes per pixel (plane q = channels 8q .. 8q+7): ldmatrix row
// addresses of 8 consecutive pixels are then 8 consecutive 16-byte words of one plane (conflict-free), and the plane pitch (361
// words, odd) keeps the staging stores of one pixel's 8 chunks conflict-free too.  Warp w computes output rows 2w and 2w+1 of
// every class (equal tap count per warp), the B fragments of a (tap, k-step) are read once from shared memory and used for both.
#include "common.cuh"

namespace d3fk {

constexpr int SD_THREADS = 256;
constexpr int SD_T = 32;                    // output tile: 32 x 32 pixels
constexpr int SD_S = SD_T / 2 + 3;          // 19: halo extent of dY per axis
constexpr int SD_NP = SD_S * SD_S;          // 361 pixels per plane
constexpr int SD_C = 64;                    // dY channels
constexpr int SD_WROW = 49 * SD_C + 8;      // bf16 per weight row (ci): +8 puts the three rows in different banks
constexpr size_t SD_SMEM = (size_t)8 * SD_NP * 16 + (size_t)3 * SD_WROW * 2;

__device__ __forceinline__ void sd_ldmatrix_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void sd_mma_bf16(float* c, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

__global__ void __launch_bounds__(SD_THREADS) stem_dgrad_mma_kernel(const __nv_bfloat16* __restrict__ dy, int ldy,
                                                                   const __nv_bfloat16* __restrict__ w, float* __restrict__ out,
                                                                   int H, int W, int Cout) {
  extern __shared__ uint4 sd_smem[];
  uint4* tile = sd_smem;                                                     // [8 planes][19][19]
  __nv_bfloat16* wsm = reinterpret_cast<__nv_bfloat16*>(tile + 8 * SD_NP);   // [3][SD_WROW]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  // weights do not depend on the previous kernel: staged before griddepcontrol.wait; rows ci >= Cout are zero
  for (int i = tid; i < 3 * 49 * SD_C / 8; i += SD_THREADS) {
    const int ci = i / (49 * SD_C / 8), k = i - ci * (49 * SD_C / 8);
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (ci < Cout) v = __ldg(reinterpret_cast<const uint4*>(w + (long long)ci * 49 * SD_C) + k);
    *reinterpret_cast<uint4*>(wsm + ci * SD_WROW + k * 8) = v;
  }
  pdl_enter();
  const int Hy = H >> 1, Wy = W >> 1;
  const int tiles_w = W / SD_T, tiles_h = H / SD_T;
  int b = blockIdx.x;
  const int tw = b % tiles_w; b /= tiles_w;
  const int th = b % tiles_h; b /= tiles_h;
  const int h0 = th * SD_T, w0 = tw * SD_T;
  const int y0 = h0 / 2 - 1, x0 = w0 / 2 - 1;                               // dY coordinates of halo pixel (0, 0)
  // stage: 8 consecutive threads load the 8 16-byte chunks of one dY pixel (128 contiguous bytes)
  constexpr int NV = 8 * SD_NP;
#pragma unroll 4
  for (int i = tid; i < NV; i += SD_THREADS) {
    const int q = i & 7, pix = i >> 3;
    const int r = pix / SD_S, c = pix - r * SD_S;
    const int gy = y0 + r, gx = x0 + c;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if ((unsigned)gy < (unsigned)Hy && (unsigned)gx < (unsigned)Wy)
      v = __ldg(reinterpret_cast<const uint4*>(dy + ((long long)(b * Hy + gy) * Wy + gx) * ldy) + q);
    tile[q * SD_NP + pix] = v;
  }
  __syncthreads();
  const uint32_t tile_s = (uint32_t)__cvta_generic_to_shared(tile);
  // ldmatrix.x4 row addresses: lanes 0-7 / 8-15 / 16-23 / 24-31 -> (pixels 0-7, plane 2ks) / (8-15, 2ks) / (0-7, 2ks+1) / (8-15, 2ks+1)
  const int lrow = (lane >> 4) * SD_NP + ((lane >> 3) & 1) * 8 + (lane & 7);
  const uint32_t* wsm32 = reinterpret_cast<const uint32_t*>(wsm);
  const long long plane = (long long)H * W;
#pragma unroll 1
  for (int cls = 0; cls < 4; ++cls) {
    const int ph = cls >> 1, pw = cls & 1;
    const int nth = 3 + ph, ntw = 3 + pw;                                    // taps per axis: kh = (1 - ph) + 2a, a < nth
    float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    const int i_lo = 2 * warp;                                               // class rows i_lo, i_lo + 1
#pragma unroll 1
    for (int a = 0; a < nth; ++a) {
      const int kh = 1 - ph + 2 * a;
#pragma unroll 1
      for (int bb = 0; bb < ntw; ++bb) {
        const int kw = 1 - pw + 2 * bb;
        // output (h0 + ph + 2i, w0 + pw + 2j) reads dY (h0/2 + i + ph + 1 - a, w0/2 + j + pw + 1 - bb) = halo (i + ph + 2 - a, j + pw + 2 - bb)
        const int col0 = pw + 2 - bb;
        const uint32_t* wt = wsm32 + ((kh * 7 + kw) * SD_C) / 2;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          uint32_t b0 = 0u, b1 = 0u;
          if (g < 3) {
            b0 = wt[g * (SD_WROW / 2) + ks * 8 + t];
            b1 = wt[g * (SD_WROW / 2) + ks * 8 + t + 4];
          }
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            const int row = i_lo + r + ph + 2 - a;
            uint32_t a0, a1, a2, a3;
            sd_ldmatrix_x4(tile_s + (uint32_t)((2 * ks * SD_NP + row * SD_S + col0 + lrow) * 16), a0, a1, a2, a3);
            sd_mma_bf16(acc[r], a0, a1, a2, a3, b0, b1);
          }
        }
      }
    }
    // C fragment: acc[r][0] / [1] = (pixel j = g, ci = 2t / 2t+1), [2] / [3] = (pixel g + 8, same ci)
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int h = h0 + ph + 2 * (i_lo + r);
      float* o = out + (long long)b * Cout * plane + (long long)h * W + w0 + pw + 2 * g;
      if (2 * t < Cout) {
        o[(2 * t) * plane] = acc[r][0];
        o[(2 * t) * plane + 16] = acc[r][2];
      }
      if (2 * t + 1 < Cout) {
        o[(2 * t + 1) * plane] = acc[r][1];
        o[(2 * t + 1) * plane + 16] = acc[r][3];
      }
    }
  }
}

// 1 = launched, 0 = not this kernel's shape (the caller falls through to the generic paths), < 0 = error
int try_launch_stem_dgrad(const d3fk_conv_params* p, cudaStream_t s) {
#ifdef D3FK_DEBUG
  static int enabled = -1;
  if (enabled < 0) { const char* v = getenv("D3FK_STEM_DGRAD"); enabled = v ? atoi(v) : 1; }
  if (!enabled) return 0;
#endif
  if (p->dtype != D3FK_BF16 || p->mode != 1 || p->kh != 7 || p->kw != 7 || p->stride != 2 || p->pad != 3) return 0;
  if (p->c0 != SD_C || p->c1 != 0 || p->up0 != 0 || p->src1 || p->Cout < 1 || p->Cout > 3) return 0;
  if (!p->out_nchw || p->out || p->res || p->stats || p->relu || p->scale || p->shift || p->bw_x) return 0;
  if (p->Ho != 2 * p->Hi || p->Wo != 2 * p->Wi || (p->Ho % SD_T) || (p->Wo % SD_T) || (p->ld0 % 8)) return 0;
  if (((uintptr_t)p->src0 & 15) || ((uintptr_t)p->w & 15)) return 0;
  const long long blocks = (long long)p->B * (p->Ho / SD_T) * (p->Wo / SD_T);
  if (blocks >= (1ll << 31)) return 0;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(stem_dgrad_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SD_SMEM);
    if (e != cudaSuccess) return set_error(D3FK_ERR_CUDA, "stem dgrad smem attribute: %s", cudaGetErrorString(e));
    attr_set = true;
  }
  launch_k(stem_dgrad_mma_kernel, dim3((unsigned)blocks), dim3(SD_THREADS), SD_SMEM, s, dim3(1, 1, 1), (const __nv_bfloat16*)p->src0,
           p->ld0, (const __nv_bfloat16*)p->w, p->out_nchw, p->Ho, p->Wo, p->Cout);
  count_launch();
  const int rc = check_launch("stem_dgrad");
  return rc ? rc : 1;
}

}  // namespace d3fk
