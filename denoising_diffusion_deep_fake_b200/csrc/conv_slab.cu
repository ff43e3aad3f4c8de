// conv_slab.cu — the slab convolution (3x3 / stride 1, Cin <= 128, W >= 16): see the comment above conv_slab_kernel.
#include "tc_common.cuh"

namespace d3fk {

// ------------------------------------------------------------------------------------------
// Slab convolution: 3x3 / stride 1 / pad 1, one source, Cin in {16, 32, 64}, W in {16, 32, 64} (forward and dgrad).
// The implicit-GEMM kernels above re-read every activation pixel once per tap (9x) from L2.  Here a persistent CTA owns
// super-tiles of S*R full image rows (S sub-tiles of R*W = 128 pixels).  For each super-tile ONE TMA box per horizontal
// tap offset (3 boxes: columns shifted by -1/0/+1, S*R+2 rows, hardware zero fill for the halo) lands in shared memory;
// all 9 taps of all S sub-tiles are then UMMA operands that differ only by a row offset into those slabs, and the 9 weight
// tiles stay resident in shared memory for the whole kernel.  L2 -> SM traffic per pixel drops from 9x to 3*(S*R+2)/(S*R)
// and no thread computes an address: warp 5 issues 3 TMA loads per super-tile, warp 4 issues the MMAs, warps 0-3 only run
// the epilogue (double-buffered TMEM accumulators), so load, MMA and epilogue of consecutive super-tiles overlap.
struct SlabSched {
  int W, H, R, S;         // image extent; rows per 128-pixel sub-tile; sub-tiles per super-tile
  int Wt, wtiles;         // tile width min(W, 128) and tiles across the image width
  int row_bytes;          // Cin * 2 = bytes of one pixel row of the K-major operand = TMA / UMMA swizzle span (32/64/128)
  int slab_bytes;         // (S*R + 2) * W * row_bytes rounded up to 1 KB
  int slab_tx;            // bytes one slab load delivers
  int stages;             // slab pipeline depth
  int w_tile_bytes;       // BN * row_bytes: one tap's resident weight tile
  int total, tiles_per_img;
  int sgn;                // +1 forward taps, -1 transposed (dgrad)
  int ksteps;             // channels per chunk / 16
  int chunks, ctot;       // 64-channel chunks per tap when Cin > 64 (each chunk is one pipeline stage); total Cin
  uint32_t layout;        // UMMA smem-descriptor layout type: 2 = SWIZZLE_128B, 4 = 64B, 6 = 32B
  int M;                  // B*H*W
  // FLAT variant (flat != 0): ONE slab per stage instead of three column-shifted ones.  The slab is the (RT + 2) x Wp
  // pixel box (Wp = Wt + 2: one halo column on each side, zero filled by TMA at the image border) kept as a flat list of
  // pixel rows; an M tile is 128 CONSECUTIVE slab positions q = r * Wp + w, so that tap (kh, kw) of every row of the tile
  // is the same flat offset kh * Wp + kw — a start-address shift of the UMMA descriptor by whole pixel rows (not a
  // multiple of the 8-row swizzle atom; measured: no descriptor base offset is needed, the swizzle follows the absolute
  // shared-memory address).  The two halo positions
  // per image row compute junk that the epilogue drops; activations are read 1.3x instead of 3.75x.
  int flat, Wp, RT;       // RT: image rows per super-tile
  uint32_t ablate;        // -DD3FK_DEBUG builds only (D3FK_SLAB_ABLATE): 1 = no epilogue work, 2 = no MMAs, 4 = no TMA data
  FastDiv dWp;
};

__device__ __forceinline__ uint64_t make_smem_desc_sw(uint32_t saddr, uint32_t sbo_bytes, uint32_t layout) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;                              // leading byte offset (unused for swizzled K-major): 16 B
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;   // stride between 8-row groups
  d |= (uint64_t)1 << 46;                              // descriptor version (Blackwell)
  d |= (uint64_t)layout << 61;
  return d;
}

// Warps: 0-7 epilogue, 8 TMA producer, 9..9+NW-1 MMA issuers: MMA warp w (w < S) issues the 9*KSTEPS*chunks MMAs of
// sub-tile w of every super-tile from ONE elected thread (elect.sync: descriptor words live in uniform registers, ~2 SASS
// instructions per MMA).  (Until round 2 the issue loop ran behind a lane compare and cost ~31 instructions per MMA — one
// MMA per ~90 cycles — which is why the taps of a sub-tile used to be split over several warps with partial accumulators
// that the epilogue had to add up.)
// Eight epilogue warps: the epilogue is a dependent chain per warp (tcgen05.ld -> convert -> store -> statistics) and with
// four warps it alone took 85 % of a narrow layer's time (ablation: D3FK_SLAB_ABLATE=6).  A warp may read TMEM lanes
// 32*(warp%4)..+32 only, so warps e and e+4 share a row quarter and split the work: the two column halves of a tile
// (BN >= 32: also halves the per-thread statistics registers) or alternate sub-tiles (BN = 16: a thread keeps a whole
// 32-byte output row).
template <int BN> struct SlabCfg {
  static constexpr int NW = BN >= 128 ? 2 : 4;
  static constexpr int EPI_WARPS = 8;
  static constexpr int THREADS = (EPI_WARPS + 1 + NW) * 32;
  static constexpr int ACC = BN < 32 ? 32 : BN;
  static constexpr int TMEM_COLS = 2 * NW * ACC;       // double buffered
};
// AFF: the epilogue applies scale / shift (eval: folded BatchNorm; head: bias) staged in shared memory.  A template
// parameter, not a run-time branch: the staging code costs the training-mode kernels 20 registers and 5-12 % of their time.
template <int BN, int KSTEPS, bool AFF>
__global__ void __launch_bounds__(SlabCfg<BN>::THREADS) conv_slab_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                                                               EpiTC e, SlabSched ss, FastDiv dWo, FastDiv dHo, int* errflag) {
  constexpr int ACC = SlabCfg<BN>::ACC;
  constexpr int NW = SlabCfg<BN>::NW;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w_base = base;                                         // [9 taps][chunks][BN rows][row_bytes]
  const uint32_t w_bytes = (uint32_t)((9 * ss.chunks * ss.w_tile_bytes + 1023) & ~1023);
  const uint32_t slab_base = base + w_bytes;                            // [stages][3][slab_bytes]
  const uint32_t stage_bytes = (ss.flat ? 1u : 3u) * ss.slab_bytes;
  const uint32_t bar_base = slab_base + ss.stages * stage_bytes;        // full[4], empty[4], acc_full[2], acc_empty[2], wbar
  uint8_t* gen_bar = smem_raw + (bar_base - smem_u32(smem_raw));
  volatile uint32_t* tmem_ptr_slot = reinterpret_cast<volatile uint32_t*>(gen_bar + 8 * 13);
  float* s_stat = reinterpret_cast<float*>(gen_bar + 128);              // [8 warps][2][BN]
  float* s_aff = s_stat + 16 * BN;                                       // [2][BN] staged scale / shift (eval: folded BN; head: bias)
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (4 + s); };
  auto acc_full_bar = [&](int b) { return bar_base + 8u * (8 + b); };
  auto acc_empty_bar = [&](int b) { return bar_base + 8u * (10 + b); };
  const uint32_t wbar = bar_base + 8u * 12;

  const int tid = threadIdx.x, warp = warp_index_uniform(), lane = tid & 31;
  const bool do_stats = e.stats != nullptr;
  const int S = ss.S;
  constexpr uint32_t tmem_cols = (uint32_t)SlabCfg<BN>::TMEM_COLS;

  if (tid == 0) {
    for (int s = 0; s < 4; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), S);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(acc_full_bar(b), S);
      mbar_init(acc_empty_bar(b), 256);
    }
    mbar_init(wbar, 1);
    fence_barrier_init();
  }
  if (tid < 256) {
    for (int i = tid; i < 16 * BN; i += 256) s_stat[i] = 0.f;
  }
  if (warp == 8 && elect_one_sync()) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    const int cchp = ss.row_bytes >> 1;   // weights are not produced by the previous kernel: warm L2 during the PDL prologue
    for (int t = 0; t < 9; ++t)
      for (int c = 0; c < ss.chunks; ++c) tma_prefetch_l2_2d(&tmB, t * ss.ctot + c * cchp, 0);
  }
  if (warp == 9) tmem_alloc(smem_u32((const void*)tmem_ptr_slot), tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = *tmem_ptr_slot;
  pdl_enter();

  if (warp == 8) {
    // ===================== TMA producer =====================
    if (elect_one_sync()) {
      // resident weights: 9 * chunks boxes {chunk channels, BN} of the packed [Cout][9*Cin] matrix (rows >= Cout zero filled)
      mbar_arrive_expect_tx(wbar, 9u * ss.chunks * ss.w_tile_bytes);
      const int cch = ss.row_bytes >> 1;
      for (int t = 0; t < 9; ++t)
        for (int c = 0; c < ss.chunks; ++c)
          tma_load_2d(w_base + (t * ss.chunks + c) * ss.w_tile_bytes, &tmB, t * ss.ctot + c * cch, 0, wbar);
      const int rows = ss.flat ? ss.RT : S * ss.R;
      // pipeline position over (super-tile, chunk) pairs as running counters: stage index, parity of the round, and whether
      // the ring has wrapped (a run-time `it % stages` / `it / stages` is a ~20-instruction sequence in every role's loop)
      int st = 0;
      uint32_t round_par = 0;
      bool wrapped = false;
      for (int t = blockIdx.x; t < ss.total; t += gridDim.x) {
        const int n = t / ss.tiles_per_img;
        const int rem = t - n * ss.tiles_per_img;
        const int hb = rem / ss.wtiles;
        const int h0 = hb * rows, w0 = (rem - hb * ss.wtiles) * ss.Wt;
        for (int c = 0; c < ss.chunks; ++c) {
          if (wrapped) mbar_wait(empty_bar(st), round_par ^ 1u, errflag);
#ifdef D3FK_DEBUG
          if (ss.ablate & 4u) {
            mbar_arrive_expect_tx(full_bar(st), 0u);
          } else
#endif
          if (ss.flat) {
            mbar_arrive_expect_tx(full_bar(st), (uint32_t)ss.slab_tx);
            tma_load_4d(slab_base + st * stage_bytes, &tmA, c * cch, w0 - 1, h0 - 1, n, full_bar(st));
          } else {
            mbar_arrive_expect_tx(full_bar(st), 3u * ss.slab_tx);
            for (int sx = 0; sx < 3; ++sx)
              tma_load_4d(slab_base + st * stage_bytes + sx * ss.slab_bytes, &tmA, c * cch, w0 + sx - 1, h0 - 1, n, full_bar(st));
          }
          if (++st == ss.stages) { st = 0; round_par ^= 1u; wrapped = true; }
        }
      }
    }
    __syncwarp();
  } else if (warp >= 9) {
    // ===================== MMA issuers =====================
    // One elected thread per sub-tile.  Every descriptor is (constant high word, low word = constant | address >> 4).
    const int w = warp - 9;                             // this warp's sub-tile
    if (w < S && elect_one_sync()) {
      constexpr uint32_t idesc = make_idesc(TC_BM, BN, 0, 0);
      const uint32_t sbo = 8u * ss.row_bytes;
      const uint64_t dtempl = make_smem_desc_sw(0, sbo, ss.layout);
      const uint32_t dhi = (uint32_t)(dtempl >> 32), dlo = (uint32_t)dtempl;
      const uint32_t img_row16 = (uint32_t)(ss.Wt * ss.row_bytes) >> 4;  // one image row of the slab, in 16-byte units
      uint32_t a_off[9], b_lo[9];
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        const int kh = tap / 3, kw = tap - kh * 3;
        const int sy = ss.sgn > 0 ? kh : 2 - kh;
        const int sx = ss.sgn > 0 ? kw : 2 - kw;
        // flat variant: the swizzle is a function of the absolute shared-memory address, so a start address shifted by whole
        // pixel rows needs no descriptor base offset (measured on B200 for SWIZZLE_32B / 64B / 128B)
        a_off[tap] = ss.flat ? ((uint32_t)((w * TC_BM + sy * ss.Wp + sx) * ss.row_bytes) >> 4)
                             : ((uint32_t)(sx * ss.slab_bytes) >> 4) + (uint32_t)(sy + w * ss.R) * img_row16;
        b_lo[tap] = dlo | ((w_base + (uint32_t)(tap * ss.chunks * ss.w_tile_bytes)) >> 4);
      }
      const uint32_t wchunk16 = (uint32_t)ss.w_tile_bytes >> 4;
      mbar_wait(wbar, 0, errflag);
      uint32_t tile_it = 0;
      int st = 0;
      uint32_t round_par = 0;
      for (int t = blockIdx.x; t < ss.total; t += gridDim.x, ++tile_it) {
        const uint32_t abuf = tile_it & 1;
        if (tile_it >= 2) mbar_wait(acc_empty_bar(abuf), ((tile_it >> 1) - 1) & 1, errflag);
        tc_fence_after();
        const uint32_t d_addr = tmem_d + abuf * (uint32_t)(NW * ACC) + (uint32_t)(w * ACC);
        uint32_t first = 0u;
        for (int c = 0; c < ss.chunks; ++c) {
          mbar_wait(full_bar(st), round_par, errflag);
          tc_fence_after();
          const uint32_t sub_lo = dlo | ((slab_base + st * stage_bytes) >> 4);
          const uint32_t bc = (uint32_t)c * wchunk16;
#ifdef D3FK_DEBUG
          if (!(ss.ablate & 2u))
#endif
          {
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
#pragma unroll
              for (int kk = 0; kk < KSTEPS; ++kk) {
                umma_f16_lohi(d_addr, sub_lo + a_off[tap] + 2u * kk, dhi, b_lo[tap] + bc + 2u * kk, dhi, idesc, first);
                first = 1u;
              }
            }
          }
          umma_commit(empty_bar(st));
          if (++st == ss.stages) { st = 0; round_par ^= 1u; }
        }
        umma_commit(acc_full_bar(abuf));
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue warps (0-7) =====================
    const int q = warp & 3, h = warp >> 2;              // TMEM lane quarter (= row group) and work half of this warp
    constexpr bool SPLIT_COLS = BN >= 32;               // halves = column halves; BN = 16: halves = alternate sub-tiles
    constexpr int NC = SPLIT_COLS ? BN / 2 : BN;        // accumulator columns of a sub-tile this warp handles
    constexpr int CW = NC >= 32 ? 32 : 16;              // columns per tcgen05.ld
    const int c_lo = SPLIT_COLS ? h * NC : 0;
    const int s_first = SPLIT_COLS ? 0 : h, s_step = SPLIT_COLS ? 1 : 2;
    // Narrow slices (16 columns per warp) keep their batch statistics in registers: a thread owns one row of every sub-tile
    // it handles, so it accumulates its own per-column sums over the whole kernel and the rows are folded ONCE at the end
    // (instead of a shuffle transpose-reduce per tile).
    constexpr bool REG_STATS = NC <= 16;
    constexpr bool affine = AFF;
    if (affine) {                    // after griddepcontrol.wait: whatever produced scale / shift has completed
      if (tid < BN) {
        s_aff[tid] = e.scale ? (tid < e.Cout ? __ldg(e.scale + tid) : 0.f) : 1.f;
        s_aff[BN + tid] = tid < e.Cout ? __ldg(e.shift + tid) : 0.f;
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
    }
    float rs[REG_STATS ? NC : 1], rq[REG_STATS ? NC : 1];
#pragma unroll
    for (int i = 0; i < (REG_STATS ? NC : 1); ++i) { rs[i] = 0.f; rq[i] = 0.f; }
    uint32_t it = 0;
    const int row = q * 32 + lane;
    float* my_stat = s_stat + warp * 2 * BN;
    for (int t = blockIdx.x; t < ss.total; t += gridDim.x, ++it) {
      const uint32_t abuf = it & 1;
      const int n = t / ss.tiles_per_img;
      const int rem = t - n * ss.tiles_per_img;
      const int hb = rem / ss.wtiles;
      const int h0 = hb * (ss.flat ? ss.RT : S * ss.R), w0 = (rem - hb * ss.wtiles) * ss.Wt;
      mbar_wait(acc_full_bar(abuf), (it >> 1) & 1, errflag);
      tc_fence_after();
#ifdef D3FK_DEBUG
      if (ss.ablate & 1u) {
        tc_fence_before();
        mbar_arrive(acc_empty_bar(abuf));
        continue;
      }
#endif
      for (int s = s_first; s < S; s += s_step) {
        long long m;
        bool row_ok;
        int on = 0, oh = 0, ow = 0;
        if (ss.flat) {
          // slab position p = r * Wp + w of this accumulator row; the columns w >= Wt are the halo positions (junk)
          const uint32_t pos = (uint32_t)(s * TC_BM + row);
          const int r = (int)fdiv(pos, ss.dWp);
          const int w = (int)pos - r * ss.Wp;
          row_ok = w < ss.Wt && r < ss.RT && h0 + r < ss.H && w0 + w < ss.W;
          m = ((long long)n * ss.H + h0 + r) * ss.W + w0 + w;
          on = n; oh = h0 + r; ow = w0 + w;
        } else {
          m = ((long long)n * ss.H + h0 + s * ss.R) * ss.W + w0 + row;   // 128 consecutive pixels
          row_ok = m < ss.M;
          if (e.out_nchw && row_ok) {
            const uint32_t pq = fdiv((uint32_t)m, dWo);
            ow = (int)m - (int)pq * e.Wo;
            on = (int)fdiv(pq, dHo);
            oh = (int)pq - on * e.Ho;
          }
        }
        // (Tried and dropped: software-pipelining the TMEM reads — the next chunk's tcgen05.ld in flight while this one is
        // stored: the extra chunk iterations and register pressure cost more than the exposed load latency.)
#pragma unroll
        for (int cl = 0; cl < NC; cl += CW) {
          const int cc = c_lo + cl;                     // first accumulator column of this chunk
          uint32_t raw[CW];
          const uint32_t taddr = tmem_d + ((uint32_t)(q * 32) << 16) + abuf * (uint32_t)(NW * ACC) + (uint32_t)(s * ACC + cc);
          // wide layers: plain batch statistics from tensor memory in the 16x256b arrangement (tmem_col_stats); the flat
          // variant (junk halo positions inside a row quarter) and the dgrad-fused BN-backward sums keep the row-wise path
          const bool tstats = !REG_STATS && do_stats && !e.bw_x && !ss.flat;
          if (tstats) {
            const long long mq = ((long long)n * ss.H + h0 + s * ss.R) * ss.W + w0 + q * 32;   // first row of this quarter
            const long long lim = (long long)ss.M - mq;
            tmem_col_stats<CW>(taddr, lim > 32 ? 32 : (int)lim, my_stat + cc, my_stat + BN + cc, lane);
          }
          if (CW == 32) tmem_ld32(taddr, raw); else tmem_ld16(taddr, raw);
          tmem_ld_wait();
          float f[CW];
#pragma unroll
          for (int i = 0; i < CW; ++i) f[i] = __uint_as_float(raw[i]);
          epilogue_chunk<CW>(f, e, m, row_ok, cc, on, oh, ow, do_stats && !REG_STATS && !tstats, my_stat + cc, my_stat + BN + cc, lane,
                             affine ? s_aff + cc : nullptr, BN);
          if (REG_STATS && do_stats) {
            if (e.bw_x) {
              float sq[CW];
              bw_stat_terms<CW>(f, sq, e, m, row_ok, cc);
#pragma unroll
              for (int i = 0; i < CW; ++i) { rs[cl + i] += f[i]; rq[cl + i] += sq[i]; }
            } else if (row_ok) {
#pragma unroll
              for (int i = 0; i < CW; ++i) { rs[cl + i] += f[i]; rq[cl + i] = fmaf(f[i], f[i], rq[cl + i]); }
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(acc_empty_bar(abuf));
    }
    if (do_stats) {
      if (REG_STATS) {                                  // NC == CW == 16
        float a[CW], b[CW];
#pragma unroll
        for (int i = 0; i < CW; ++i) { a[i] = rs[i]; b[i] = rq[i]; }
        const float cs = warp_colsum16(a, lane), cq = warp_colsum16(b, lane);
        if (lane < CW) {
          my_stat[c_lo + lane] = cs;
          my_stat[BN + c_lo + lane] = cq;
        }
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (tid < BN && tid < e.Cout) {
        float a = 0.f, b = 0.f;
#pragma unroll
        for (int wq = 0; wq < 8; ++wq) { a += s_stat[wq * 2 * BN + tid]; b += s_stat[wq * 2 * BN + BN + tid]; }
        atomicAdd(&e.stats[tid], (double)a);
        atomicAdd(&e.stats[e.Cout + tid], e.bw_x ? bw_second_sum((double)a, (double)b, e, tid) : (double)b);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 9) tmem_dealloc(tmem_d, tmem_cols);
}

static int g_use_slab = 1;   // D3FK_SLAB=0: never take the slab path
static int g_slab_flat = 0;        // flat (single-slab) variant — 1: whenever W >= min_w; 0: only for sizes the three-slab layout
                                   // cannot take (ragged W / H); -1: never.  Correct for every swizzle width, but measured NOT
                                   // faster than the three-slab layout on B200 (these kernels are not load-bound)
static int g_slab_flat_min_w = 32; // narrower images: the halo positions would waste too many accumulator rows
static int g_slab_ablate = 0;      // D3FK_SLAB_ABLATE (debug builds): SlabSched::ablate

// Slab-path eligibility and geometry.  Returns false when the generic kernels must be used.
static bool slab_plan(const Gather& g, const d3fk_conv_params* p, int BN, SlabSched& ss, int& smem) {
  if (!g_use_slab) return false;
  if (p->kh != 3 || p->kw != 3 || p->stride != 1 || p->pad != 1 || p->c1 != 0 || p->up0 != 0) return false;
  if (p->Ho != p->Hi || p->Wo != p->Wi) return false;
  const int C = g.ctot, W = p->Wi, H = p->Hi;
  if (C != 16 && C != 32 && C != 64 && C != 128) return false;   // 128 = two 64-channel chunks (one pipeline stage each)
  if (p->Cout > BN || (!p->out_nchw && p->Cout != BN)) return false;
  if (((uintptr_t)p->src0 & 15) || (g.ld0 % 8)) return false;
  const int cch = C > 64 ? 64 : C;
  ss.chunks = C / cch;
  ss.ctot = C;
  ss.row_bytes = cch * 2;
  ss.layout = cch == 64 ? 2u : cch == 32 ? 4u : 6u;
  ss.ksteps = cch / 16;
  ss.w_tile_bytes = BN * ss.row_bytes;
  ss.sgn = p->mode ? -1 : 1;
  ss.M = g.M;
  ss.ablate = (uint32_t)g_slab_ablate;
  const int w_bytes = (9 * ss.chunks * ss.w_tile_bytes + 1023) & ~1023;
  const int NW = BN >= 128 ? 2 : 4;                    // MMA warps (SlabCfg<BN>::NW): S must divide it
  const int Wt_l = W < TC_BM ? W : TC_BM;
  const bool legacy_ok = (W == 16 || W == 32 || W == 64 || W % 128 == 0) && H % (TC_BM / Wt_l) == 0;
  if ((g_slab_flat > 0 || (g_slab_flat == 0 && !legacy_ok)) && W >= g_slab_flat_min_w) {
    // FLAT variant: one (RT + 2) x (Wt + 2) slab per stage, M tiles over consecutive slab positions (see SlabSched).  Any
    // H and W: ragged tiles are masked in the epilogue, out-of-image rows / columns are TMA zero fill.
    const int Wt = W < TC_BM ? W : TC_BM, Wp = Wt + 2;
    ss.W = W; ss.H = H; ss.Wt = Wt; ss.Wp = Wp; ss.wtiles = cdiv(W, Wt); ss.R = 1;
    ss.flat = 1; ss.dWp = make_fastdiv((uint32_t)Wp);
    for (int S = NW; S >= 1; S >>= 1) {
      const int rt_max = (S * TC_BM - Wt) / Wp + 1;   // last valid position (RT - 1) * Wp + Wt - 1 < S * 128
      if (S * TC_BM < Wt || rt_max < 1) continue;
      const int T = cdiv(H, rt_max), RT = cdiv(H, T);     // balanced row split of the image
      const int used = cdiv((RT - 1) * Wp + Wt, TC_BM);    // sub-tiles that hold valid positions
      if (S > 1 && used <= S / 2) continue;                // a smaller super-tile does the same work
      const int rows_loaded = (RT + 2) * Wp;
      const int rows_read = S * TC_BM + 2 * Wp + 2;        // the furthest (junk) row a tap of the last sub-tile touches
      const int slab = ((rows_loaded > rows_read ? rows_loaded : rows_read) * ss.row_bytes + 1023) & ~1023;
      for (int stages = 4; stages >= 2; --stages) {
        const int need = 1024 + w_bytes + stages * slab + 128 + 18 * BN * 4;
        if (need > SLAB_MAX_SMEM) continue;
        ss.S = S; ss.RT = RT;
        ss.slab_bytes = slab;
        ss.slab_tx = rows_loaded * ss.row_bytes;
        ss.stages = stages;
        ss.tiles_per_img = T * ss.wtiles;
        ss.total = p->B * ss.tiles_per_img;
        smem = need;
        return true;
      }
    }
    ss.flat = 0;
  }
  if (W != 16 && W != 32 && W != 64 && (W % 128)) return false;
  const int Wt = W < TC_BM ? W : TC_BM;
  const int R = TC_BM / Wt;
  if (H % R) return false;
  ss.W = W; ss.H = H; ss.R = R; ss.Wt = Wt; ss.wtiles = W / Wt;
  // largest super-tile whose double-buffered accumulators fit TMEM and whose 2-stage slabs fit shared memory
  for (int S = NW; S >= 1; S >>= 1) {
    if (H % (S * R)) continue;
    const int slab = ((S * R + 2) * Wt * ss.row_bytes + 1023) & ~1023;
    for (int stages = 3; stages >= 2; --stages) {
      const int need = 1024 + w_bytes + stages * 3 * slab + 128 + 18 * BN * 4;
      if (need > SLAB_MAX_SMEM) continue;
      ss.S = S;
      ss.slab_bytes = slab;
      ss.slab_tx = (S * R + 2) * Wt * ss.row_bytes;
      ss.stages = stages;
      ss.tiles_per_img = (H / (S * R)) * ss.wtiles;
      ss.total = p->B * ss.tiles_per_img;
      smem = need;
      return true;
    }
  }
  return false;
}

template <int BN, int KSTEPS, bool AFF>
static int launch_conv_slab_bn(const Gather& g, const d3fk_conv_params* p, cudaStream_t s, const SlabSched& ss, int smem) {
  EpiTC e{(bf16*)p->out, p->out_nchw, p->scale, p->shift, (const bf16*)p->res, p->stats, p->ldo, p->ldr, p->relu, p->Cout, p->Ho, p->Wo,
           (const bf16*)p->bw_x, (const bf16*)p->bw_act, p->bw_mean, p->bw_invstd, p->bw_ldx, p->bw_ldact, p->bw_relu};
  alignas(64) CUtensorMap tmA, tmB;
  const int C = g.ctot;
  {
    uint64_t dims[2] = {(uint64_t)g.K, (uint64_t)p->Cout};
    uint64_t strides[1] = {(uint64_t)g.K * 2};
    uint32_t bx[2] = {(uint32_t)(ss.row_bytes >> 1), (uint32_t)BN};
    int rc = get_tensor_map(&tmB, p->w, 2, dims, strides, bx, ss.row_bytes);
    if (rc) return rc;
  }
  {
    uint64_t dims[4] = {(uint64_t)C, (uint64_t)g.Wi, (uint64_t)g.Hi, (uint64_t)g.B};
    uint64_t strides[3] = {(uint64_t)g.ld0 * 2, (uint64_t)g.Wi * g.ld0 * 2, (uint64_t)g.Hi * g.Wi * g.ld0 * 2};
    uint32_t bx[4] = {(uint32_t)(ss.row_bytes >> 1), (uint32_t)ss.Wt, (uint32_t)(ss.S * ss.R + 2), 1u};
    if (ss.flat) { bx[1] = (uint32_t)ss.Wp; bx[2] = (uint32_t)(ss.RT + 2); }
    int rc = get_tensor_map(&tmA, p->src0, 4, dims, strides, bx, ss.row_bytes);
    if (rc) return rc;
  }
  int occ = (227 * 1024) / (smem + 1024);
  const int tmem_cols = SlabCfg<BN>::TMEM_COLS;
  if (occ * tmem_cols > 512) occ = 512 / tmem_cols;
  if (occ < 1) occ = 1;
  int grid = ss.total < g_num_sms * occ ? ss.total : g_num_sms * occ;
  // epi: as the conv_tc line (0 plain, 2 BN-backward sums, 3 affine / bias: the AFF variant); the slab kernel has no fused BN
  const int epi = p->bw_x ? 2 : AFF ? 3 : 0;
  if (g_verbose) fprintf(stderr, "[d3fk] slab<%d> mode=%d M=%d C=%d Cout=%d W=%d S=%d stages=%d smem=%d grid=%d total=%d flat=%d RT=%d epi=%d\n", BN, g.mode, g.M, C, p->Cout, ss.W, ss.S, ss.stages, smem, grid, ss.total, ss.flat, ss.RT, epi);
  launch_k(conv_slab_kernel<BN, KSTEPS, AFF>, dim3(grid), dim3(SlabCfg<BN>::THREADS), (size_t)smem, s, dim3(1, 1, 1), tmA, tmB, e, ss,
           make_fastdiv((uint32_t)g.Wo), make_fastdiv((uint32_t)g.Ho), g_dev_error_flag);
  count_launch();
  return check_launch("conv_slab");
}

// returns 1 when the slab path took the op, 0 when it is not eligible, < 0 on error
int try_launch_conv_slab(const Gather& g, const d3fk_conv_params* p, cudaStream_t s) {
  const int C = p->Cout;
  const int BN = C <= 16 ? 16 : C <= 32 ? 32 : C <= 64 ? 64 : C <= 128 ? 128 : 0;
  if (!BN) return 0;
  if (p->out_nchw && BN != 16) return 0;
  SlabSched ss;
  memset(&ss, 0, sizeof(ss));
  int smem = 0;
  if (!slab_plan(g, p, BN, ss, smem)) return 0;
  int rc;
  const bool aff = p->scale != nullptr || p->shift != nullptr;
#define SLAB_CASE(bn, ks)                                                                                     \
  if (BN == bn && ss.ksteps == ks) rc = aff ? launch_conv_slab_bn<bn, ks, true>(g, p, s, ss, smem)            \
                                            : launch_conv_slab_bn<bn, ks, false>(g, p, s, ss, smem); else
  SLAB_CASE(16, 1) SLAB_CASE(16, 2) SLAB_CASE(16, 4) SLAB_CASE(32, 1) SLAB_CASE(32, 2) SLAB_CASE(32, 4)
  SLAB_CASE(64, 1) SLAB_CASE(64, 2) SLAB_CASE(64, 4) SLAB_CASE(128, 1) SLAB_CASE(128, 2) SLAB_CASE(128, 4)
  rc = set_error(D3FK_ERR_UNSUPPORTED, "slab: BN=%d ksteps=%d", BN, ss.ksteps);
#undef SLAB_CASE
  return rc ? rc : 1;
}


int slab_init() {
  cudaError_t e = cudaSuccess;
#ifdef D3FK_DEBUG
  if (const char* v = getenv("D3FK_SLAB")) g_use_slab = atoi(v);
  if (const char* v = getenv("D3FK_SLAB_FLAT")) g_slab_flat = atoi(v);
  if (const char* v = getenv("D3FK_SLAB_FLAT_MIN_W")) g_slab_flat_min_w = atoi(v);
  if (const char* v = getenv("D3FK_SLAB_ABLATE")) g_slab_ablate = atoi(v);
#endif
  D3FK_SET_SMEM((conv_slab_kernel<16, 1, false>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<16, 1, true>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<16, 2, false>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<16, 2, true>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<16, 4, false>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<16, 4, true>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<32, 1, false>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<32, 1, true>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<32, 2, false>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<32, 2, true>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<32, 4, false>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<32, 4, true>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<64, 1, false>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<64, 1, true>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<64, 2, false>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<64, 2, true>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<64, 4, false>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<64, 4, true>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<128, 1, false>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<128, 1, true>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<128, 2, false>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<128, 2, true>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<128, 4, false>), SLAB_MAX_SMEM)
  D3FK_SET_SMEM((conv_slab_kernel<128, 4, true>), SLAB_MAX_SMEM)
  if (e != cudaSuccess) return set_error(D3FK_ERR_CUDA, "cudaFuncSetAttribute (slab): %s", cudaGetErrorString(e));
  return D3FK_OK;
}

}  // namespace d3fk
