// conv_tc.cu — bf16 implicit-GEMM convolution and dgrad on the Blackwell 5th-gen tensor cores (the weight gradients live
// in wgrad_tc.cu, the narrow 3x3 layers in conv_slab.cu): tcgen05.mma issued by one ELECTED thread (elect.sync),
// accumulators double-buffered in TMEM, operands in 128B-swizzled shared memory — by TMA boxes (PATH 2: stride-1 "same"
// convolutions; also the space-to-depth stem, conv mode 2) or by an asynchronous per-thread gather (PATH 0 / 1: cp.async
// completing on mbarriers) —, tcgen05.ld epilogue fused with BN statistics / folded-BN affine / residual / ReLU, split K
// over a thread-block cluster with an st.async reduce-scatter, train-mode BatchNorm fused behind a grid barrier.
//
// D[M = B*Ho*Wo pixels, N = Cout] = A[M, K = taps*Cin] x W[N, K]^T     (both K-major)
//
// Warp roles (320 threads): warps 0-3 = gather producers (PATH 0 / 1), then epilogue (TMEM lane quarter = warp % 4);
// warp 4 = TMEM allocator + MMA issuer; warp 5 = TMA producer; warps 6-9 = epilogue helpers (odd column chunks).
#include "tc_common.cuh"

namespace d3fk {

// Pipeline depth.  In the eval forward (FUSE 3: the sampler) 128-wide tiles fed by TMA (PATH 2) run ONE CTA per SM with six
// stages (198 KB): a single CTA needs ~200 KB in flight to cover latency x bandwidth of the L2 -> SM operand stream
// (layer3-size tile: 14.3 -> 12.6 us, sampling step 0.896 -> 0.863 ms).  Training keeps three stages / two CTAs per SM:
// measured 3.77 -> 3.83 ms per step with six — a 198 KB CTA leaves no room for a weight-gradient CTA of the side stream
// next to it, and that overlap is worth more than the faster main loop.
template <int BN, int PATH, int FUSE> struct ConvCfg {
  static constexpr int STAGES = BN >= 128 ? ((PATH == 2 && FUSE == 3) ? 6 : 3) : 4;
  static constexpr int B_STAGE_BYTES = BN * 128;
  static constexpr int SMEM = 1024 + STAGES * (A_STAGE_BYTES + B_STAGE_BYTES) + 256 + 10 * BN * 4;
  static constexpr int ACC_COLS = BN < 32 ? 32 : BN;   // one accumulator buffer
  static constexpr int TMEM_COLS = 2 * ACC_COLS;        // double buffered: epilogue of tile i overlaps MMAs of tile i+1
};

// Tile schedule.  KS == 1: tile t -> (m tile, n tile), consecutive CTAs walk consecutive m tiles, persistent loop.
// KS > 1 (split K over a thread-block cluster of KS CTAs): one tile per CTA, t -> (k split = cluster rank, m tile, n tile);
// the KS partial accumulators are reduce-scattered through distributed shared memory (no workspace, no second kernel).
struct TileSched {
  int MT, NT, KS, kb_per_split, nkb, total, a_ca;
  int bw, bh, bn, wt, ht;   // PATH 2: the 128-pixel M tile as a (w, h, n) box and the tile grid along w / h
  int off_w, off_h;         // PATH 2: box origin offsets (-pad forward, +pad transposed; windowed rows: 0 / -pad)
  int a_pitch;              // PATH 2: pixels per image row of the A tensor in memory (0: Wi; windowed rows: Wi + 3)
};

__device__ __forceinline__ void decode_tile(const TileSched& ts, int t, int& mt, int& nt, int& ks) {
  if (ts.KS > 1) {
    ks = t % ts.KS;
    const int r = t / ts.KS;
    mt = r % ts.MT;
    nt = r / ts.MT;
  } else {
    ks = 0;
    mt = t % ts.MT;
    nt = t / ts.MT;
  }
}

// Fused train-mode BatchNorm (forward): when every output tile of the layer is resident at once (one tile per CTA, the
// accumulator parked in TMEM — or, for split-K clusters, the reduced slice in shared memory), the conv kernel itself
// finalises the batch statistics behind a grid-wide barrier and applies normalise + residual + ReLU from the fp32
// accumulator: raw conv output (kept for the backward pass) and activation are both written by this one kernel and the
// separate BN kernel (launch, prologue, a re-read of the raw tensor) disappears.
struct FuseBN {
  const float* gamma; const float* beta;
  float* mean; float* invstd; float* running_mean; float* running_var; long long* nbt;
  float* scale; float* shift;   // published for the backward pass (d3fk_bn_params.mask_from_x)
  bf16* act; const bf16* res;
  unsigned* barrier;         // zeroed by the forward's statistics memset
  long long count;
  int ldact, ldr, relu;
  float eps, momentum;
};

// PATH 0 (LINEAR): one source, no upsample, forward gather or stride-1 transposed gather — the tap
//   offset is the same for every row, so a row costs two compares, one 64-bit add and the cp.async.
// PATH 1 (GENERIC): nearest-2x upsample + channel concat (decoder conv1) and stride-2 transposed gather.
// PATH 2 (TMA): stride-1 "same" convolutions with Cin % 64 == 0 and power-of-two extents: the A tile of tap (kh,kw)
//   is the NHWC box {64 channels, bw, bh, bn} shifted by the tap offset, loaded by ONE cp.async.bulk.tensor.4d with
//   hardware zero fill for the padding halo — no per-thread address arithmetic at all.
// The weight tile is always a TMA 2-D box {64, BN} of the packed [Cout][K] matrix (OOB rows / K tail zero filled).
template <int BN, int PATH, int FUSE>
__global__ void __launch_bounds__(TC_THREADS, 2) conv_tc_kernel(Gather g, FastDiv dWo, FastDiv dHo, const __grid_constant__ CUtensorMap tmA,
                                                             const __grid_constant__ CUtensorMap tmB, EpiTC e, TileSched ts,
                                                             FuseBN fb, int* errflag) {
  using Cfg = ConvCfg<BN, PATH, FUSE>;
  constexpr int STAGES = Cfg::STAGES;
  constexpr int CW = BN >= 32 ? 32 : 16;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t a_base = base;
  const uint32_t b_base = base + STAGES * A_STAGE_BYTES;
  const uint32_t bar_base = b_base + STAGES * Cfg::B_STAGE_BYTES;  // full[S], empty[S], acc_full[2], acc_empty[2], tmem ptr
  uint8_t* gen_bar = smem_raw + (base - smem_u32(smem_raw)) + STAGES * (A_STAGE_BYTES + Cfg::B_STAGE_BYTES);
  volatile uint32_t* tmem_ptr_slot = reinterpret_cast<volatile uint32_t*>(gen_bar + 8 * (2 * STAGES + 4));
  float* s_stat = reinterpret_cast<float*>(gen_bar + 256);  // [4 warps][2][BN]
  float* s_aff = s_stat + 8 * BN;                           // [2][BN] scale / shift of the current n tile (see epilogue_chunk)
  constexpr bool affine = FUSE == 3;        // FUSE 3: plain convolution whose epilogue applies staged scale / shift (eval)
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto acc_full_bar = [&](int b) { return bar_base + 8u * (2 * STAGES + b); };
  auto acc_empty_bar = [&](int b) { return bar_base + 8u * (2 * STAGES + 2 + b); };
  const uint32_t recv_bar = bar_base + 8u * (2 * STAGES + 5);   // split K: the partial tiles of the cluster have landed here

  const int tid = threadIdx.x, warp = warp_index_uniform(), lane = tid & 31;
  // Epilogue warps: 0-3 (also the gather producers of PATH 0/1) and the helpers 6-9.  A warp may touch TMEM lanes
  // 32*(warp%4)..+32 only, so helper warp w shares the lane quarter of primary warp w%4 and takes every other column
  // chunk: the epilogue is a dependent instruction chain per warp (~1 us per 32 columns with one warp per scheduler).
  const bool is_epi = warp < 4 || warp >= 6;
  const int q = warp & 3;                         // TMEM lane quarter / row group of this epilogue warp
  const int half = warp >= 6 ? 1 : 0;             // helpers take the odd column chunks
  const int etid = warp < 4 ? tid : 128 + (tid - 192);   // 0..255 over the 8 epilogue warps
  // (re)stage the affine coefficients of n tile `nt`: all 8 epilogue warps call it at the same point of their tile loops
  auto stage_affine = [&](int nt, bool live) {
    asm volatile("bar.sync 1, 256;" ::: "memory");     // nobody still reads the previous tile's coefficients
    const int ch = nt * BN + etid;
    if (etid < BN) {                                   // (warm pass: no global loads before griddepcontrol.wait)
      s_aff[etid] = e.scale ? (live && ch < e.Cout ? __ldg(e.scale + ch) : 0.f) : 1.f;
      s_aff[BN + etid] = live && ch < e.Cout ? __ldg(e.shift + ch) : 0.f;
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
  };
  const bool clus = ts.KS > 1;
  const bool do_stats = e.stats != nullptr;
  TL_DECL
  TL_BEGIN

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), PATH == 2 ? 1 : 129);   // 128 gather threads + the TMA thread's expect_tx arrive
      mbar_init(empty_bar(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(acc_full_bar(b), 1);
      mbar_init(acc_empty_bar(b), EPI_THREADS);
    }
    mbar_init(recv_bar, 1);
    fence_barrier_init();
  }
  if (is_epi) {
    for (int i = etid; i < 8 * BN; i += EPI_THREADS) s_stat[i] = 0.f;
  }
  if (warp == 5 && elect_one_sync()) {
    tma_prefetch_desc(&tmB);
    if (PATH == 2) tma_prefetch_desc(&tmA);
    // The packed weights are not written by the preceding kernel (pack_all ran at the start of the step), so the first
    // pipeline stages' weight tiles are pulled into L2 now, while the previous kernel is still draining (PDL prologue).
    int mt0, nt0, ks0;
    decode_tile(ts, blockIdx.x, mt0, nt0, ks0);
    const int kbp = ks0 * ts.kb_per_split;
    for (int i = 0; i < STAGES && kbp + i < ts.nkb; ++i) tma_prefetch_l2_2d(&tmB, (kbp + i) * TC_BK, nt0 * BN);
  }
  if (FUSE == 2 && is_epi && e.bw_x) {
    // Fused BN-backward reduction: the epilogue reads one row segment of the forward's raw output / activation per lane.
    // They were written a whole forward ago (HBM, not L2) and not by the preceding kernel: pull the first tile's segments
    // into L2 now, so the loads on the epilogue's dependent chain are L2 hits.
    int mt0, nt0, ks0;
    decode_tile(ts, blockIdx.x, mt0, nt0, ks0);
    const long long mp = (long long)mt0 * TC_BM + q * 32 + lane;
    if (mp < g.M) {
      for (int b = half * 128; b < BN * 2; b += 256) {
        prefetch_l2(reinterpret_cast<const char*>(e.bw_x + mp * e.bw_ldx + nt0 * BN) + b);
        if (e.bw_relu) prefetch_l2(reinterpret_cast<const char*>(e.bw_act + mp * e.bw_ldact + nt0 * BN) + b);
      }
    }
  }
  if (warp == 4) tmem_alloc(smem_u32((const void*)tmem_ptr_slot), Cfg::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = *tmem_ptr_slot;
  if (tid == 0) { TL_STAMP(1) }
  // No griddepcontrol.wait here: every role executes pdl_enter() itself, the epilogue warps only AFTER a dry run of their
  // code (see "warm pass" below) — so far nothing has touched memory the previous kernel writes.

  // flush this CTA's accumulated statistics of n tile `nt` (epilogue warps only)
  auto flush_stats = [&](int nt) {
    asm volatile("bar.sync 1, 256;" ::: "memory");
    const int n0 = nt * BN;
    if (tid < BN && n0 + tid < e.Cout) {
      const float a = (s_stat[tid] + s_stat[2 * BN + tid]) + (s_stat[4 * BN + tid] + s_stat[6 * BN + tid]);
      const float b = (s_stat[BN + tid] + s_stat[3 * BN + tid]) + (s_stat[5 * BN + tid] + s_stat[7 * BN + tid]);
      if (a != 0.f || b != 0.f) {
        atomicAdd(&e.stats[n0 + tid], (double)a);
        atomicAdd(&e.stats[e.Cout + n0 + tid], (FUSE == 2 && e.bw_x) ? bw_second_sum((double)a, (double)b, e, n0 + tid) : (double)b);
      }
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    for (int i = etid; i < 8 * BN; i += EPI_THREADS) s_stat[i] = 0.f;
    asm volatile("bar.sync 1, 256;" ::: "memory");
  };

  // FUSE: after this CTA's statistics are flushed — grid barrier, then scale / shift of the tile's BN channels into s_stat
  // (free again after the flush): s_stat[c] = scale, s_stat[BN + c] = shift.  The CTA with m tile 0 (and k slice 0)
  // publishes mean / invstd / running statistics of its n tile.
  auto fuse_finalize = [&](int nt, bool publisher) {
    asm volatile("bar.sync 1, 256;" ::: "memory");
    if (tid == 0) grid_barrier_arrive_wait(fb.barrier, gridDim.x, errflag);
    asm volatile("bar.sync 1, 256;" ::: "memory");
    const int ch = nt * BN + tid;
    if (tid < BN && ch < e.Cout) {
      const double n = (double)fb.count;
      const double mean = __ldcg(e.stats + ch) / n;
      double var = __ldcg(e.stats + e.Cout + ch) / n - mean * mean;
      if (var < 0) var = 0;
      const double invstd = rsqrt(var + (double)fb.eps);
      const double gm = (double)__ldg(fb.gamma + ch), bt = (double)__ldg(fb.beta + ch);
      s_stat[tid] = (float)(gm * invstd);
      s_stat[BN + tid] = (float)(bt - mean * gm * invstd);
      if (publisher) {
        fb.mean[ch] = (float)mean;
        fb.invstd[ch] = (float)invstd;
        if (fb.scale) { fb.scale[ch] = s_stat[tid]; fb.shift[ch] = s_stat[BN + tid]; }
        if (fb.running_mean) {
          const double unbiased = n > 1 ? var * n / (n - 1) : var;
          fb.running_mean[ch] = (float)((1.0 - fb.momentum) * fb.running_mean[ch] + fb.momentum * mean);
          fb.running_var[ch] = (float)((1.0 - fb.momentum) * fb.running_var[ch] + fb.momentum * unbiased);
        }
        if (ch == 0 && fb.nbt) *fb.nbt += 1;
      }
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
  };
  // FUSE: activation of CWF accumulator columns [ct, ct + CWF) (tile-relative) of output row m
  auto fuse_apply = [&](float* f, int ncol, long long m, bool row_ok, int nt, int ct) {
    if (!row_ok) return;
    const int cbase = nt * BN + ct;
    for (int q = 0; q < ncol / 8; ++q) {
      float y[8];
#pragma unroll
      for (int i = 0; i < 8; ++i)      // from the bf16-ROUNDED raw value: bit-identical to the two-kernel form (and to the backward's mask)
        y[i] = fmaf(__bfloat162float(__float2bfloat16_rn(f[q * 8 + i])), s_stat[ct + q * 8 + i], s_stat[BN + ct + q * 8 + i]);
      if (fb.res) {
        const uint4 rr = __ldg(reinterpret_cast<const uint4*>(fb.res + m * fb.ldr + cbase + q * 8));
        const bf16* rb16 = reinterpret_cast<const bf16*>(&rr);
#pragma unroll
        for (int i = 0; i < 8; ++i) y[i] += __bfloat162float(rb16[i]);
      }
      if (fb.relu) {
#pragma unroll
        for (int i = 0; i < 8; ++i) y[i] = fmaxf(y[i], 0.f);
      }
      uint4 o;
      __nv_bfloat162* o2 = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
      for (int i = 0; i < 4; ++i) o2[i] = __floats2bfloat162_rn(y[2 * i], y[2 * i + 1]);
      *reinterpret_cast<uint4*>(fb.act + m * fb.ldact + cbase + q * 8) = o;
    }
  };

  if (warp == 5) {
    // ===================== TMA producer (one elected thread) =====================
    pdl_enter();   // the prologue above overlapped the previous kernel; from here on its results are visible
    if (tid == 160) { TL_STAMP(2) }
    if (elect_one_sync()) {
      uint32_t kbg = 0;
      const int sgn = g.mode ? -1 : 1;
      for (int t = blockIdx.x; t < ts.total; t += gridDim.x) {
        int mt, nt, ks;
        decode_tile(ts, t, mt, nt, ks);
        const int kb0 = ks * ts.kb_per_split;
        const int kb1 = min(ts.nkb, kb0 + ts.kb_per_split);
        int w0 = 0, h0 = 0, i0 = 0, tap = 0, c = 0, khi = 0, kwi = 0;
        if (PATH == 2) {
          const int tw = mt % ts.wt;
          const int r2 = mt / ts.wt;
          w0 = tw * ts.bw + ts.off_w;
          h0 = (r2 % ts.ht) * ts.bh + ts.off_h;
          i0 = (r2 / ts.ht) * ts.bn;
          const int k = kb0 * TC_BK;
          tap = k / g.ctot;
          c = k - tap * g.ctot;
          khi = tap / g.kw;
          kwi = tap - khi * g.kw;
        }
        for (int kb = kb0; kb < kb1; ++kb, ++kbg) {
          const int s = kbg % STAGES;
          if (kbg >= STAGES) mbar_wait(empty_bar(s), ((kbg / STAGES) - 1) & 1, errflag);
          mbar_arrive_expect_tx(full_bar(s), Cfg::B_STAGE_BYTES + (PATH == 2 ? A_STAGE_BYTES : 0));
          tma_load_2d(b_base + s * Cfg::B_STAGE_BYTES, &tmB, kb * TC_BK, nt * BN, full_bar(s));
          if (PATH == 2) {
            tma_load_4d(a_base + s * A_STAGE_BYTES, &tmA, c, w0 + sgn * kwi, h0 + sgn * khi, i0, full_bar(s));
            c += TC_BK;
            if (c >= g.ctot) {
              c = 0;
              if (++kwi == g.kw) { kwi = 0; ++khi; }
            }
          }
        }
      }
    }
    __syncwarp();
    if (clus) cluster_sync_relaxed();   // this warp's arrival at the cluster barrier (the epilogue warps arrive from their branch)
  } else if (warp == 4) {
    // ===================== MMA issuer (one elected thread) =====================
    pdl_enter();
    if (elect_one_sync()) {
      constexpr uint32_t idesc = make_idesc(TC_BM, BN, 0, 0);
      uint32_t kbg = 0, tile_iter = 0;
      for (int t = blockIdx.x; t < ts.total; t += gridDim.x, ++tile_iter) {
        int mt, nt, ks;
        decode_tile(ts, t, mt, nt, ks);
        const int kb0 = ks * ts.kb_per_split;
        const int kb1 = min(ts.nkb, kb0 + ts.kb_per_split);
        const uint32_t abuf = tile_iter & 1;
        if (tile_iter >= 2) {   // the epilogue must have drained this accumulator buffer (two tiles ago)
          mbar_wait(acc_empty_bar(abuf), ((tile_iter >> 1) - 1) & 1, errflag);
          tc_fence_after();
        }
        const uint32_t d_addr = tmem_d + abuf * Cfg::ACC_COLS;
        for (int kb = kb0; kb < kb1; ++kb, ++kbg) {
          const int s = kbg % STAGES;
          mbar_wait(full_bar(s), (kbg / STAGES) & 1, errflag);
          if (kbg == 0) { TL_STAMP(3) }
          tc_fence_after();
          const uint32_t a_addr = a_base + s * A_STAGE_BYTES;
          const uint32_t b_addr = b_base + s * Cfg::B_STAGE_BYTES;
#pragma unroll
          for (int kk = 0; kk < TC_BK / 16; ++kk) {
            uint64_t ad = make_smem_desc(a_addr + kk * 32, 16, 1024);
            uint64_t bd = make_smem_desc(b_addr + kk * 32, 16, 1024);
            umma_f16(d_addr, ad, bd, idesc, (kb > kb0 || kk > 0) ? 1u : 0u);
          }
          umma_commit(empty_bar(s));
        }
        umma_commit(acc_full_bar(abuf));
        TL_STAMP(4)
      }
    }
    __syncwarp();
    if (clus) cluster_sync_relaxed();
  } else {
    // ===================== epilogue warps (0-3: also the gather producers of PATH 0 / 1; 6-9) =====================
    // WARM PASS.  A kernel of this step lives for 10-20 us and most of its code runs exactly once per CTA: the epilogue
    // (and the split-K reduction) used to execute at ~10 cycles per instruction, two thirds of the stall samples being
    // "no instruction" — cold instruction fetches from L2 (ncu source page; phase stamps: 7.8 us from the last MMA to the
    // end of the epilogue of a split-K tile).  So the epilogue warps first run their whole code path DRY — before
    // griddepcontrol.wait, i.e. while the previous kernel is still draining: no barrier waits, row_ok = false (no global
    // load / store), no remote shared-memory store — which pulls the instructions into the SM's instruction cache; the live
    // pass then runs at cache-hit speed.  `pass` is opaque to the compiler: ONE copy of the code serves both passes.
    const int j = tid & 7;    // 16-byte chunk (8 channels) within the 128-byte k-row
    const int rb = tid >> 3;  // rows rb + 16*i
    const uint32_t sw = (uint32_t)((j ^ (rb & 7)) << 4);
    const int sgn = g.mode ? -1 : 1;
    const uint32_t smask = g.mode ? (uint32_t)(g.stride - 1) : 0u;   // transposed gather: coordinate must be a multiple
    const int sshift = g.mode ? g.sshift : 0;                        // of the stride (forward folds it into h0/w0)
    const int row = q * 32 + lane;
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
      int pass_v = pass;
      asm volatile("" : "+r"(pass_v));
      const bool live = pass_v != 0;
      if (live) {
        pdl_enter();
        if (tid == 0) { TL_STAMP(2) }
      }
      uint32_t kbg = 0;  // k-blocks issued by this CTA so far (pipeline stage / phase bookkeeping)
      uint32_t tile_iter = 0;
      int cur_nt = -1, cur_aff_nt = -1;
      for (int t = blockIdx.x; t < ts.total; t += gridDim.x, ++tile_iter) {
        int mt, nt, ks;
        decode_tile(ts, t, mt, nt, ks);
        const int m0 = mt * TC_BM, n0 = nt * BN;
        const int kb0 = ks * ts.kb_per_split;
        const int kb1 = min(ts.nkb, kb0 + ts.kb_per_split);

        if (PATH != 2 && warp < 4 && live) {
          // ---- per-row state
          int rh[8], rw[8];
          int rn[8];                    // GENERIC: image index
          const bf16* rp[8];            // LINEAR: pointer of (n, h0, w0, channel 0) in src0
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int m = m0 + rb + 16 * i;
            int n = 0, h0 = -(1 << 28), w0 = 0;
            if (m < g.M) {
              const uint32_t qq = fdiv((uint32_t)m, dWo);
              const int wo = m - (int)qq * g.Wo;
              n = (int)fdiv(qq, dHo);
              const int ho = (int)qq - n * g.Ho;
              if (g.mode == 0) { h0 = ho * g.stride - g.pad; w0 = wo * g.stride - g.pad; }
              else { h0 = ho + g.pad; w0 = wo + g.pad; }
            }
            rh[i] = h0; rw[i] = w0;
            if (PATH == 0) rp[i] = (const bf16*)g.src0 + ((long long)(n * g.Hi + h0) * g.Wi + w0) * g.ld0;
            else rn[i] = n;
          }
          // ---- k state of this thread's chunk at the first k-block of the split
          int k = kb0 * TC_BK + j * 8;
          int tap = k / g.ctot;
          int c = k - tap * g.ctot;
          int khi = tap / g.kw, kwi = tap - khi * g.kw;

          for (int kb = kb0; kb < kb1; ++kb, ++kbg) {
            const int s = kbg % STAGES;
            if (kbg >= STAGES) mbar_wait(empty_bar(s), ((kbg / STAGES) - 1) & 1, errflag);
            const bool k_ok = k < g.K;
            const uint32_t a_dst = a_base + s * A_STAGE_BYTES + rb * 128 + sw;
            const int dkh = sgn * khi, dkw = sgn * kwi;
            if (PATH == 0) {
              const long long koff = (long long)(dkh * g.Wi + dkw) * g.ld0 + c;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const bool ok = k_ok && (unsigned)(rh[i] + dkh) < (unsigned)g.Hi && (unsigned)(rw[i] + dkw) < (unsigned)g.Wi;
                const void* src = ok ? (const void*)(rp[i] + koff) : g.src0;
                if (ts.a_ca) cp_async_16_ca(a_dst + i * (16 * 128), src, ok ? 16u : 0u);
                else cp_async_16(a_dst + i * (16 * 128), src, ok ? 16u : 0u);
              }
            } else {
              const bool second = c >= g.c0;
              const bf16* sb = second ? (const bf16*)g.src1 + (c - g.c0) : (const bf16*)g.src0 + c;
              const int ld = second ? g.ld1 : g.ld0;
              const int up = second ? 0 : g.up0;
              const int hs = g.Hi >> up, wsz = g.Wi >> up;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const int th = rh[i] + dkh, tw = rw[i] + dkw;
                const int hi = th >> sshift, wi = tw >> sshift;
                const bool ok = k_ok && (((uint32_t)(th | tw)) & (0x80000000u | smask)) == 0 && hi < g.Hi && wi < g.Wi;
                const long long pix = (long long)((rn[i] * hs + (hi >> up)) * wsz + (wi >> up));
                const void* src = ok ? (const void*)(sb + pix * ld) : g.src0;
                if (ts.a_ca) cp_async_16_ca(a_dst + i * (16 * 128), src, ok ? 16u : 0u);
                else cp_async_16(a_dst + i * (16 * 128), src, ok ? 16u : 0u);
              }
            }
            cp_async_mbar_arrive(full_bar(s));
            mbar_arrive(full_bar(s));
            k += TC_BK;
            c += TC_BK;
            while (c >= g.ctot) {
              c -= g.ctot;
              if (++kwi == g.kw) { kwi = 0; ++khi; }
            }
          }
        }

        // ===================== epilogue: TMEM -> registers -> global =====================
        const uint32_t abuf = tile_iter & 1;
        if (live) {
          mbar_wait(acc_full_bar(abuf), (tile_iter >> 1) & 1, errflag);
          if (tid == 0) { TL_STAMP(5) }
          tc_fence_after();
        }
        const int m = m0 + row;
        const bool row_ok = live && m < g.M;
        if (!clus) {
          if (affine && (cur_aff_nt != nt || !live)) {
            stage_affine(nt, live);
            cur_aff_nt = live ? nt : -1;
          }
          if (live && do_stats && cur_nt != nt) {
            if (cur_nt >= 0) flush_stats(cur_nt);
            cur_nt = nt;
          }
          int on = 0, oh = 0, ow = 0;
          if (e.out_nchw && row_ok) {
            const uint32_t qq = fdiv((uint32_t)m, dWo);
            ow = m - (int)qq * e.Wo;
            on = (int)fdiv(qq, dHo);
            oh = (int)qq - on * e.Ho;
          }
#pragma unroll 1
          for (int cc = half * CW; cc < BN; cc += 2 * CW) {
            uint32_t raw[CW];
            const uint32_t taddr = tmem_d + ((uint32_t)(q * 32) << 16) + abuf * Cfg::ACC_COLS + (uint32_t)cc;
            // plain batch statistics (training forward): from tensor memory in the 16x256b arrangement, BEFORE the stores
            const bool tstats = do_stats && !(FUSE == 2 && e.bw_x);
            if (tstats) tmem_col_stats<CW>(taddr, live ? g.M - (m0 + q * 32) : 0, s_stat + q * 2 * BN + cc, s_stat + q * 2 * BN + BN + cc, lane);
            if (CW == 32) tmem_ld32(taddr, raw); else tmem_ld16(taddr, raw);
            tmem_ld_wait();
            float f[CW];
#pragma unroll
            for (int i = 0; i < CW; ++i) f[i] = __uint_as_float(raw[i]);
            epilogue_chunk<CW, FUSE == 2>(f, e, (long long)m, row_ok, n0 + cc, on, oh, ow, do_stats && !tstats, s_stat + q * 2 * BN + cc,
                                          s_stat + q * 2 * BN + BN + cc, lane, affine ? s_aff + cc : nullptr, BN);
            if (tid == 0 && cc == 0) { TL_STAMP(8) }
          }
          if (tid == 0) { TL_STAMP(9) }
          if (FUSE == 1 && live) {
            // one tile per CTA (the launcher guarantees it): statistics -> grid barrier -> activation from the parked accumulator
            flush_stats(nt);
            cur_nt = -1;
            fuse_finalize(nt, mt == 0);
#pragma unroll 1
            for (int cc = half * CW; cc < BN; cc += 2 * CW) {
              uint32_t raw[CW];
              const uint32_t taddr = tmem_d + ((uint32_t)(q * 32) << 16) + abuf * Cfg::ACC_COLS + (uint32_t)cc;
              if (CW == 32) tmem_ld32(taddr, raw); else tmem_ld16(taddr, raw);
              tmem_ld_wait();
              float f[CW];
#pragma unroll
              for (int i = 0; i < CW; ++i) f[i] = __uint_as_float(raw[i]);
              fuse_apply(f, CW, (long long)m, row_ok, nt, cc);
            }
          }
          if (live) {
            tc_fence_before();   // this tile's TMEM reads are done: hand the accumulator buffer back to the MMA issuer
            mbar_arrive(acc_empty_bar(abuf));
          }
        } else {
          // ===================== split-K reduction across the cluster (KS CTAs, one k slice each) =====================
          // Every CTA holds a 128 x BN fp32 partial tile in TMEM.  Column slice j (SL = BN/KS columns) is owned by rank j:
          // each CTA writes its partial of slice j into slot [own rank] of rank j's receive buffer (the pipeline stages are
          // dead once every CTA has finished its main loop), then each owner sums KS slots and runs the epilogue on its slice.
          // The partials travel as st.async stores that count their bytes on the OWNER's mbarrier: the only cluster-wide
          // barrier is the (relaxed) "all main loops done"; an owner starts its epilogue as soon as its own 128 x BN x 4
          // bytes have landed.  (Before: barrier.cluster release / acquire around the scatter — a MEMBAR.ALL.GPU per arrive
          // and everyone waiting for the slowest scatter of the cluster: 4-5 us from the last MMA to the epilogue.)
          const int KS = ts.KS, SL = BN / KS, sl4 = SL >> 2;
          const uint32_t rank = cluster_ctarank();
          const uint32_t recv = a_base;   // [KS][SL/4][128 rows] float4
          if (live) {
            if (etid == 0) mbar_arrive_expect_tx(recv_bar, (uint32_t)(TC_BM * BN * 4));
            tc_fence_before();
            cluster_sync_relaxed();         // all main loops done (every epilogue warp saw acc_full): the stages are dead
            tc_fence_after();
            if (tid == 0) { TL_STAMP(11) }
          }
#pragma unroll 1
          for (int cc = half * CW; cc < BN; cc += 2 * CW) {
            uint32_t raw[CW];
            const uint32_t taddr = tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)cc;
            if (CW == 32) tmem_ld32(taddr, raw); else tmem_ld16(taddr, raw);
            tmem_ld_wait();
#pragma unroll
            for (int q4 = 0; q4 < CW / 4; ++q4) {
              const int col = cc + 4 * q4;
              const int owner = col / SL, within = col - owner * SL;
              const uint32_t la = recv + (uint32_t)((((int)rank * sl4 + (within >> 2)) * 128 + row) * 16);
              const uint32_t ra = mapa_shared(la, (uint32_t)owner);
              if (live) st_async_f4(ra, raw[4 * q4], raw[4 * q4 + 1], raw[4 * q4 + 2], raw[4 * q4 + 3], mapa_shared(recv_bar, (uint32_t)owner));
            }
          }
          if (live) {
            if (tid == 0) { TL_STAMP(12) }
            mbar_wait(recv_bar, 0, errflag);   // all KS partials of my slice have landed (complete_tx of the st.async stores)
            if (tid == 0) { TL_STAMP(13) }
          }
          if (affine) stage_affine(nt, live);
          const int cslice = (int)rank * SL;     // first column of my slice within the tile
#pragma unroll 1
          for (int ch = half * 16; ch < SL; ch += 32) {
            float f[16];
#pragma unroll
            for (int c4 = 0; c4 < 4; ++c4) {
              float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
              for (int r = 0; r < KS; ++r) {
                const float4 v = ld_shared_f4(recv + (uint32_t)(((r * sl4 + (ch >> 2) + c4) * 128 + row) * 16));
                a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
              }
              f[4 * c4] = a.x; f[4 * c4 + 1] = a.y; f[4 * c4 + 2] = a.z; f[4 * c4 + 3] = a.w;
            }
            const int ct = cslice + ch;          // column within the tile
            const bool tstats = do_stats && !(FUSE == 2 && e.bw_x);
            if (tstats) {
              // park the reduced slice in (dead) tensor memory and take the statistics in the 16x256b arrangement
              const uint32_t taddr = tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)ct;
              if (live) tmem_st16(taddr, f);   // (never in the warm pass: the MMA issuer may already be accumulating)
              __syncwarp();
              tmem_col_stats<16>(taddr, live ? g.M - (m0 + q * 32) : 0, s_stat + q * 2 * BN + ct, s_stat + q * 2 * BN + BN + ct, lane);
            }
            epilogue_chunk<16, FUSE == 2>(f, e, (long long)m, row_ok, nt * BN + ct, 0, 0, 0, do_stats && !tstats, s_stat + q * 2 * BN + ct,
                                          s_stat + q * 2 * BN + BN + ct, lane, affine ? s_aff + ct : nullptr, BN);
          }
          if (tid == 0) { TL_STAMP(14) }
          if (live && do_stats) flush_stats(nt);
          if (tid == 0) { TL_STAMP(15) }
          if (FUSE == 1 && live) {
            fuse_finalize(nt, mt == 0 && rank == 0);
#pragma unroll 1
            for (int ch = half * 16; ch < SL; ch += 32) {
              float f[16];
#pragma unroll
              for (int c4 = 0; c4 < 4; ++c4) {
                float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int r = 0; r < KS; ++r) {
                  const float4 v = ld_shared_f4(recv + (uint32_t)(((r * sl4 + (ch >> 2) + c4) * 128 + row) * 16));
                  a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
                }
                f[4 * c4] = a.x; f[4 * c4 + 1] = a.y; f[4 * c4 + 2] = a.z; f[4 * c4 + 3] = a.w;
              }
              fuse_apply(f, 16, (long long)m, row_ok, nt, cslice + ch);
            }
          }
        }
        if (!live || clus) break;   // warm pass: one dry tile; split K: one tile per CTA
      }
      if (tid == 0) { TL_STAMP(10) }
      if (live && !clus && do_stats && cur_nt >= 0) flush_stats(cur_nt);
    }
  }

  if (tid == 0) { TL_STAMP(6) }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_d, Cfg::TMEM_COLS);
  if (tid == 128) { TL_STAMP(7) }
}

int g_num_sms = 148;
int g_verbose = 0;
int g_max_cluster = 8;
static int g_tile_loop = 1;   // D3FK_TILE_LOOP=0: one CTA per tile (debug aid)
static int g_a_ca = 0;        // D3FK_A_CA=1: L1-allocating activation gather
static int g_occ_cap = 0;     // D3FK_OCC=n: cap CTAs per SM
static int g_use_tma_a = 1;   // D3FK_TMA_A=0: force the gather producers (debug aid)
static int g_split_tiles = 74;  // split K only when the output tiles fill at most this many SMs
static int g_split_cta_cap = 100; // split K: tiles * KS at most this many percent of the SM count (D3FK_SPLIT_CAP, debug builds)

// Fusion request of launch_conv_bn (below): set around a launch_conv_tc call; the launcher takes it when the layer
// qualifies (BN == 128 tiles, one tile per co-resident CTA) and reports back through `taken`.
struct FuseReq { const d3fk_bn_params* bn; unsigned* barrier; bool taken; };
static thread_local FuseReq* t_fuse = nullptr;
static int g_fuse_bn = 1;   // D3FK_FUSE_BN=0: always run BatchNorm as its own kernel

template <int BN, int PATH>
static int launch_conv_tc_bn(const Gather& g, const d3fk_conv_params* p, cudaStream_t s, const TileSched& box) {
  EpiTC e{(bf16*)p->out, p->out_nchw, p->scale, p->shift, (const bf16*)p->res, p->stats, p->ldo, p->ldr, p->relu, p->Cout, p->Ho, p->Wo,
           (const bf16*)p->bw_x, (const bf16*)p->bw_act, p->bw_mean, p->bw_invstd, p->bw_ldx, p->bw_ldact, p->bw_relu};
  TileSched ts = box;
  ts.MT = cdiv(g.M, TC_BM);
  ts.NT = cdiv(p->Cout, BN);
  ts.nkb = cdiv(g.K, TC_BK);
  ts.KS = 1;
  const int tiles = ts.MT * ts.NT;
  ts.a_ca = g_a_ca && p->kh > 1;
  // split K over a cluster when the output tiles cannot fill the chip and the reduction is long
  if (BN == 128 && !p->out_nchw && p->Cout % BN == 0 && tiles <= g_split_tiles && ts.nkb >= 8 && g_max_cluster > 1) {
    int ks = 1;
    // One CTA per SM at most (tiles * KS <= SMs): the reduce-scatter moves (KS - 1) / KS of every CTA's 64 KB partial tile
    // over the SM-to-SM network, which carries ~17-21 B per cycle and SM (measured: 4 us for KS = 4 at two CTAs per SM, as
    // long as the whole main loop) — a second resident CTA doubles that traffic per SM and buys the main loop nothing
    // (it is bound by the L2 -> SM operand stream either way).
    while (ks * 2 <= g_max_cluster && ks * 2 <= 8 && tiles * ks * 2 <= g_split_cta_cap * g_num_sms / 100 && ts.nkb / (ks * 2) >= 4) ks *= 2;
    while (ks > 1 && tiles * ks > cluster_capacity(ks, 2)) ks >>= 1;
    ts.KS = ks;
  }
  ts.kb_per_split = cdiv(ts.nkb, ts.KS);
  if (ts.KS > 1 && (ts.KS - 1) * ts.kb_per_split >= ts.nkb) {   // every rank needs at least one k-block
    ts.KS = 1;
    ts.kb_per_split = ts.nkb;
  }
  ts.total = tiles * ts.KS;
  const bool eval_affine = !p->bw_x && (p->scale || p->shift);      // launches the FUSE 3 variant below
  const int smem_bytes = eval_affine ? ConvCfg<BN, PATH, 3>::SMEM : ConvCfg<BN, PATH, 0>::SMEM;
  int occ = (227 * 1024) / (smem_bytes + 1024);
  if (occ * ConvCfg<BN, PATH, 0>::TMEM_COLS > 512) occ = 512 / ConvCfg<BN, PATH, 0>::TMEM_COLS;
  if (g_occ_cap > 0 && occ > g_occ_cap) occ = g_occ_cap;
  int grid = ts.total < g_num_sms * occ ? ts.total : g_num_sms * occ;
  if (!g_tile_loop || ts.KS > 1) grid = ts.total;

  // TMA descriptors: weights [Cout][K] as a {64, BN} box; PATH 2 also the activation tensor as a 4-D NHWC box
  alignas(64) CUtensorMap tmA, tmB;
  memset(&tmA, 0, sizeof(tmA));
  {
    uint64_t dims[2] = {(uint64_t)g.K, (uint64_t)p->Cout};
    uint64_t strides[1] = {(uint64_t)g.K * 2};
    uint32_t bx[2] = {TC_BK, (uint32_t)BN};
    int rc = get_tensor_map(&tmB, p->w, 2, dims, strides, bx, 128);
    if (rc) return rc;
  }
  if (PATH == 2) {
    uint64_t dims[4] = {(uint64_t)g.c0, (uint64_t)g.Wi, (uint64_t)g.Hi, (uint64_t)g.B};
    const uint64_t pitch = (uint64_t)(ts.a_pitch ? ts.a_pitch : g.Wi);
    uint64_t strides[3] = {(uint64_t)g.ld0 * 2, pitch * g.ld0 * 2, (uint64_t)g.Hi * pitch * g.ld0 * 2};
    uint32_t bx[4] = {TC_BK, (uint32_t)ts.bw, (uint32_t)ts.bh, (uint32_t)ts.bn};
    int rc = get_tensor_map(&tmA, p->src0, 4, dims, strides, bx, 128);
    if (rc) return rc;
  }
  // fused BatchNorm: every tile resident at once (grid == tiles * KS <= co-resident capacity), 128-wide tiles only
  FuseBN fb;
  memset(&fb, 0, sizeof(fb));
  bool fuse = false;
  if (BN == 128 && t_fuse && g_fuse_bn && p->stats && !p->scale && !p->shift && !p->res && !p->relu && !p->out_nchw && p->mode == 0 &&
      p->Cout % BN == 0 && ts.total <= cluster_capacity_safe(ts.KS)) {
    const d3fk_bn_params* b = t_fuse->bn;
    fb.gamma = b->gamma; fb.beta = b->beta; fb.mean = b->mean; fb.invstd = b->invstd; fb.scale = b->scale; fb.shift = b->shift;
    fb.running_mean = b->running_mean; fb.running_var = b->running_var; fb.nbt = (long long*)b->num_batches_tracked;
    fb.act = (bf16*)b->y; fb.res = (const bf16*)b->res; fb.barrier = t_fuse->barrier; fb.count = b->count;
    fb.ldact = b->ldy; fb.ldr = b->ldr; fb.relu = b->relu; fb.eps = b->eps; fb.momentum = b->momentum;
    fuse = true;
    grid = ts.total;
    t_fuse->taken = true;
  }
  // epi = the FUSE template argument of the kernel launched below: 0 plain, 1 fused BN, 2 BN-backward sums, 3 eval affine / bias
  const int epi = p->bw_x ? 2 : fuse ? 1 : (p->scale || p->shift) ? 3 : 0;
  if (g_verbose) fprintf(stderr, "[d3fk] conv<%d,%d> mode=%d M=%d K=%d Cout=%d tiles=%d KS=%d kbps=%d grid=%d fuse=%d epi=%d\n", BN, PATH, g.mode, g.M, g.K, p->Cout, tiles, ts.KS, ts.kb_per_split, grid, (int)fuse, epi);
  cudaError_t le;
  if (p->bw_x)
    le = launch_k(conv_tc_kernel<BN, PATH, 2>, dim3(grid), dim3(TC_THREADS), ConvCfg<BN, PATH, 2>::SMEM, s, dim3(ts.KS, 1, 1), g,
                  make_fastdiv((uint32_t)g.Wo), make_fastdiv((uint32_t)g.Ho), tmA, tmB, e, ts, fb, g_dev_error_flag);
  else if (BN == 128 && fuse)
    le = launch_k(conv_tc_kernel<BN, PATH, (BN == 128 ? 1 : 0)>, dim3(grid), dim3(TC_THREADS), ConvCfg<BN, PATH, 1>::SMEM, s, dim3(ts.KS, 1, 1), g,
                  make_fastdiv((uint32_t)g.Wo), make_fastdiv((uint32_t)g.Ho), tmA, tmB, e, ts, fb, g_dev_error_flag);
  else if (p->scale || p->shift)
    le = launch_k(conv_tc_kernel<BN, PATH, 3>, dim3(grid), dim3(TC_THREADS), ConvCfg<BN, PATH, 3>::SMEM, s, dim3(ts.KS, 1, 1), g,
                  make_fastdiv((uint32_t)g.Wo), make_fastdiv((uint32_t)g.Ho), tmA, tmB, e, ts, fb, g_dev_error_flag);
  else
    le = launch_k(conv_tc_kernel<BN, PATH, 0>, dim3(grid), dim3(TC_THREADS), ConvCfg<BN, PATH, 0>::SMEM, s, dim3(ts.KS, 1, 1), g,
                  make_fastdiv((uint32_t)g.Wo), make_fastdiv((uint32_t)g.Ho), tmA, tmB, e, ts, fb, g_dev_error_flag);
  if (le != cudaSuccess) return set_error(D3FK_ERR_CUDA, "conv_tc launch: %s", cudaGetErrorString(le));
  count_launch();
  return check_launch("conv_tc");
}

template <int PATH>
static int launch_conv_tc_path(const Gather& g, const d3fk_conv_params* p, cudaStream_t s, const TileSched& box) {
  const int C = p->Cout;
  if (C <= 16) return launch_conv_tc_bn<16, PATH>(g, p, s, box);
  D3FK_CHECK_ARG(p->out_nchw == nullptr, "out_nchw only for Cout <= 16");
  if (C % 128 == 0) return launch_conv_tc_bn<128, PATH>(g, p, s, box);
  if (C % 64 == 0) return launch_conv_tc_bn<64, PATH>(g, p, s, box);
  if (C % 32 == 0) return launch_conv_tc_bn<32, PATH>(g, p, s, box);
  return set_error(D3FK_ERR_UNSUPPORTED, "conv_tc: Cout=%d (need <=16 or a multiple of 32)", C);
}

// PATH 2 eligibility: the 128-pixel M tile must be an axis-aligned (w, h, n) box whose pixel order equals the linear
// output-pixel order: bw = min(W,128) columns, then bh rows, then bn images, each level fully covered before the next.
static bool tma_box(const Gather& g, const d3fk_conv_params* p, TileSched& ts) {
  if (!g_use_tma_a) return false;
  if (p->c1 != 0 || p->up0 != 0 || p->stride != 1 || g.ctot % TC_BK != 0) return false;
  if (p->Ho != p->Hi || p->Wo != p->Wi || 2 * p->pad != p->kh - 1 || p->kh != p->kw) return false;
  if (((uintptr_t)p->src0 & 15) || (g.ld0 % 8)) return false;
  const int W = p->Wi, H = p->Hi;
  int bw = W < TC_BM ? W : TC_BM;
  if (TC_BM % bw || W % bw) return false;
  int bh = TC_BM / bw;
  if (bh > H) bh = H;
  if ((TC_BM / bw) % bh || H % bh) return false;
  int bn = TC_BM / (bw * bh);
  if (bw < W && bh != 1) return false;
  if (bh < H && bn != 1) return false;
  if (bn > 256) return false;
  ts.bw = bw; ts.bh = bh; ts.bn = bn; ts.wt = W / bw; ts.ht = H / bh;
  ts.off_w = ts.off_h = p->mode ? p->pad : -p->pad;
  ts.a_pitch = 0;
  return true;
}

// conv mode 2 ("windowed rows", include/d3fk.h): the space-to-depth stem.  Every (pixel, kh) is one contiguous 128-byte row of
// the padded space-to-depth image, so the A operand is a 4-D TMA box over a tensor map whose pixel stride (32 B) is smaller
// than its innermost extent (128 B) — overlapping windows; the kernel is the ordinary PATH 2 kernel.
static int launch_conv_windowed(const d3fk_conv_params* p, cudaStream_t s) {
  D3FK_CHECK_ARG(p->c0 == 64 && p->c1 == 0 && p->ld0 == 16 && p->kh == 4 && p->kw == 1 && p->stride == 1 && p->up0 == 0,
                 "conv mode 2: c0 = 64, ld0 = 16, 4 x 1 taps, stride 1");
  D3FK_CHECK_ARG(p->Ho == p->Hi && p->Wo == p->Wi && p->Cout == 64 && !p->out_nchw && !p->bw_x, "conv mode 2: Ho = Hi, Wo = Wi, Cout = 64");
  d3fk_conv_params q = *p;
  q.mode = 0;      // forward tap order; the window geometry lives in the tile schedule
  Gather g;
  int rc = make_gather(g, q.src0, nullptr, q.c0, 0, q.ld0, 0, 0, q.B, q.Hi, q.Wi, q.Ho, q.Wo, q.kh, q.kw, 1, q.pad, 0);
  if (rc) return rc;
  TileSched box;
  memset(&box, 0, sizeof(box));
  q.pad = 0; q.kh = q.kw = 1;          // tma_box() checks a "same" geometry: true for the window view (the taps are handled below)
  if (!tma_box(g, &q, box)) return set_error(D3FK_ERR_UNSUPPORTED, "conv mode 2: the 128-pixel tile is not a (w, h, n) box for %d x %d", p->Ho, p->Wo);
  q.pad = p->pad; q.kh = p->kh; q.kw = p->kw;
  box.off_w = 0;
  box.off_h = -p->pad;
  box.a_pitch = p->Wi + 3;
  return launch_conv_tc_bn<64, 2>(g, &q, s, box);
}

int try_launch_conv_slab(const Gather& g, const d3fk_conv_params* p, cudaStream_t s);   // conv_slab.cu
int try_launch_head_conv(const d3fk_conv_params* p, cudaStream_t s);
int try_launch_stem_dgrad(const d3fk_conv_params* p, cudaStream_t s);   // stem_dgrad.cu
int launch_conv_tc(const d3fk_conv_params* p, cudaStream_t s) {
  Gather g;
  int rc = make_gather(g, p->src0, p->src1, p->c0, p->c1, p->ld0, p->ld1, p->up0, p->B, p->Hi, p->Wi, p->Ho, p->Wo, p->kh,
                       p->kw, p->stride, p->pad, p->mode);
  if (rc) return rc;
  D3FK_CHECK_ARG(p->out || p->out_nchw, "no output");
  D3FK_CHECK_ARG(p->out_nchw || (p->ldo % 8 == 0), "ldo must be a multiple of 8");
  D3FK_CHECK_ARG(!p->scale || p->shift, "scale requires shift");
  D3FK_CHECK_ARG(((uintptr_t)p->w & 15) == 0, "weights must be 16-byte aligned");
  if (p->mode == 2) return launch_conv_windowed(p, s);
  const int head = try_launch_head_conv(p, s);          // 16 -> 3 channels, fp32 NCHW out: CUDA cores (head_conv.cu)
  if (head) return head < 0 ? head : D3FK_OK;
  const int stem = try_launch_stem_dgrad(p, s);         // 7x7 / stride-2 input gradient, 64 -> 3 channels, fp32 NCHW out
  if (stem) return stem < 0 ? stem : D3FK_OK;
  const int slab = try_launch_conv_slab(g, p, s);
  if (slab) return slab < 0 ? slab : D3FK_OK;
  TileSched box;
  memset(&box, 0, sizeof(box));
  if (tma_box(g, p, box)) return launch_conv_tc_path<2>(g, p, s, box);
  const bool linear = p->c1 == 0 && p->up0 == 0 && (p->mode == 0 || p->stride == 1);
  return linear ? launch_conv_tc_path<0>(g, p, s, box) : launch_conv_tc_path<1>(g, p, s, box);
}

// conv + train-mode BatchNorm (+residual) + ReLU as one op: fused into the conv kernel when the layer qualifies, otherwise
// the two kernels back to back (same results up to the rounding of the raw tensor the unfused BN reads back).
int launch_bn_apply(const d3fk_bn_params* p, cudaStream_t s);
int launch_conv_bn_tc(const d3fk_convbn_params* p, cudaStream_t s) {
  FuseReq req{&p->bn, (unsigned*)p->barrier, false};
  t_fuse = p->barrier ? &req : nullptr;
  int rc = launch_conv_tc(&p->conv, s);
  t_fuse = nullptr;
  if (rc || req.taken) return rc;
  return launch_bn_apply(&p->bn, s);
}


int slab_init();
int wgrad_init();
int tc_init() {
  cudaError_t e = cudaSuccess;
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0)
    g_num_sms = sms;
  if (const char* v = getenv("D3FK_VERBOSE")) g_verbose = atoi(v);   // prints launch geometry; changes nothing
#ifdef D3FK_DEBUG
  // Experiment knobs (tile scheduling, split-K cluster size, path selection).  Several of them change the summation order
  // and with it the rounding of the results, so they exist only in -DD3FK_DEBUG builds (tools/build_debug.sh), never in
  // the shipped libd3fk.so.
  if (const char* v = getenv("D3FK_TILE_LOOP")) g_tile_loop = atoi(v);
  if (const char* v = getenv("D3FK_A_CA")) g_a_ca = atoi(v);
  if (const char* v = getenv("D3FK_OCC")) g_occ_cap = atoi(v);
  if (const char* v = getenv("D3FK_TMA_A")) g_use_tma_a = atoi(v);
  if (const char* v = getenv("D3FK_SPLIT_TILES")) g_split_tiles = atoi(v);
  if (const char* v = getenv("D3FK_SPLIT_CAP")) g_split_cta_cap = atoi(v);
  if (const char* v = getenv("D3FK_CLUSTER")) g_max_cluster = atoi(v);
  if (const char* v = getenv("D3FK_FUSE_BN")) g_fuse_bn = atoi(v);
#endif
  D3FK_SET_SMEM((conv_tc_kernel<16, 0, 0>), (ConvCfg<16, 0, 0>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<32, 0, 0>), (ConvCfg<32, 0, 0>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<64, 0, 0>), (ConvCfg<64, 0, 0>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<128, 0, 0>), (ConvCfg<128, 0, 0>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<16, 1, 0>), (ConvCfg<16, 1, 0>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<32, 1, 0>), (ConvCfg<32, 1, 0>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<64, 1, 0>), (ConvCfg<64, 1, 0>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<128, 1, 0>), (ConvCfg<128, 1, 0>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<16, 2, 0>), (ConvCfg<16, 2, 0>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<32, 2, 0>), (ConvCfg<32, 2, 0>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<64, 2, 0>), (ConvCfg<64, 2, 0>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<128, 2, 0>), (ConvCfg<128, 2, 0>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<16, 0, 2>), (ConvCfg<16, 0, 2>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<16, 1, 2>), (ConvCfg<16, 1, 2>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<16, 2, 2>), (ConvCfg<16, 2, 2>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<32, 0, 2>), (ConvCfg<32, 0, 2>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<32, 1, 2>), (ConvCfg<32, 1, 2>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<32, 2, 2>), (ConvCfg<32, 2, 2>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<64, 0, 2>), (ConvCfg<64, 0, 2>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<64, 1, 2>), (ConvCfg<64, 1, 2>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<64, 2, 2>), (ConvCfg<64, 2, 2>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<128, 0, 2>), (ConvCfg<128, 0, 2>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<128, 1, 2>), (ConvCfg<128, 1, 2>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<128, 2, 2>), (ConvCfg<128, 2, 2>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<128, 0, 1>), (ConvCfg<128, 0, 1>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<128, 1, 1>), (ConvCfg<128, 1, 1>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<128, 2, 1>), (ConvCfg<128, 2, 1>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<16, 0, 3>), (ConvCfg<16, 0, 3>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<16, 1, 3>), (ConvCfg<16, 1, 3>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<16, 2, 3>), (ConvCfg<16, 2, 3>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<32, 0, 3>), (ConvCfg<32, 0, 3>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<32, 1, 3>), (ConvCfg<32, 1, 3>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<32, 2, 3>), (ConvCfg<32, 2, 3>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<64, 0, 3>), (ConvCfg<64, 0, 3>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<64, 1, 3>), (ConvCfg<64, 1, 3>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<64, 2, 3>), (ConvCfg<64, 2, 3>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<128, 0, 3>), (ConvCfg<128, 0, 3>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<128, 1, 3>), (ConvCfg<128, 1, 3>::SMEM))
  D3FK_SET_SMEM((conv_tc_kernel<128, 2, 3>), (ConvCfg<128, 2, 3>::SMEM))
  if (e != cudaSuccess) return set_error(D3FK_ERR_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  int rc = slab_init();
  if (rc) return rc;
  return wgrad_init();
}

}  // namespace d3fk
