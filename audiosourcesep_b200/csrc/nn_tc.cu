// Fused coupling network on the 5th-generation tensor cores (sm_100a).
//
// One launch evaluates ShiftAndLogScaleConvNet (flow_tfk_layers.py:73-84) for one Glow step as a
// chain of three GEMMs per 128-pixel tile, never spilling the 512-wide hidden activations to HBM:
//
//   stage 1  conv 3x3 (C/2 -> 512) as implicit GEMM: A = im2col(xb) built in shared memory by the
//            worker warps as split-bf16 [hi | lo] (K = 2*9*C/2), B = K1 (bf16)           N = 512
//   stage 2  conv 1x1 (512 -> 512): A = relu(p1) (bf16, written by the epilogue straight into the
//            SWIZZLE_128B K-major operand layout), B = diag(g1') K2                        N = 512
//   stage 3  conv 3x3 (512 -> C) as GEMM + col2im: A = relu(p2), B = [diag(g2') K3[tap]]_tap, N = 9C;
//            the 9 per-tap partial outputs G[p][tap][c] go to global memory (fp32) and a cheap
//            gather kernel sums G[p+off(tap)][tap] over the in-bounds taps ("same" zero padding,
//            with the BatchNorm offset b2' handled per tap so borders stay exact).
//
// BatchNorm runs in inference mode in the reference (SURVEY.md 8(a) row 6), so its affine is folded
// into the next GEMM's weights on the host (nn_tc_prepare).
//
// Pipeline per CTA (320 threads, persistent over tiles, 1 CTA / SM) -- see the comment above k_nn_tc4:
//   warp 0     producer: streams pre-swizzled 16-bit weight tile images (32 KB) with TMA bulk copies
//              (cp.async.bulk -> UBLKCP) into a 3-stage ring.
//   warp 1     MMA issuer: one thread issues tcgen05.mma (M=128, N<=256, K=16) with A and B
//              SWIZZLE_128B shared-memory descriptors, fp32 accumulators in TMEM (512 columns);
//              tcgen05.commit releases ring slots and signals the epilogues.
//   warps 2-9  workers: build the stage-1 operand, run the epilogues (tcgen05.ld 32x32b -> bias +
//              ReLU (+ mask bits for the backward pass) -> bf16 / fp16 -> swizzled st.shared), stage G
//              for the TMA bulk store.
//
// The data-gradient kernel is the same pipeline with transposed weights:
//   stage 1  conv3^T: A = im2col(gr) (split-bf16, K = 2*9*C), B = diag(g2') K3^T, epilogue = ReLU mask 2
//   stage 2  B = diag(g1') K2^T, epilogue = ReLU mask 1
//   stage 3  conv1^T as GEMM + col2im: B = K1 (N = 9*C/2), gather sums G'[p-off(tap)][tap].
#include "nn_tc_shared.cuh"

namespace asep {

namespace {

// ===================================================================================================
// K-pipelined kernel (default): the three GEMMs of a tile and their epilogues overlap panel by panel.
//
// Measured on B200 (tools/tc_timing.py): a tcgen05.mma with M = 128 costs max(~100, N/2) cycles, so N = 256
// instructions are the only efficient shape and the two 256-column accumulators H0 / H1 fill all of TMEM; an
// N-quarter variant with relu(p1) kept in TMEM ("TS" form, N = 128) was bit-exact but no faster.  This kernel keeps
// k_nn_tc2's layout (8 x 16 KB operand panels that hold a1, then h1, then h2 in place; 3 x 32 KB weight ring; the
// same tile-image stream) and removes the serialisation by tracking readiness per 64-column K panel:
//
//   * all 8 worker warps convert the SAME accumulator half, one 64-column panel at a time (32 columns per warp),
//     and signal panel_ready[p];
//   * S2(H0) starts when E1 has drained H0 (panels 0-3) and consumes panels 4-7 as E1 produces them;
//   * E2(H0) runs under S2(H1), writing h2 panel p over h1 panel p as soon as S2(H1) has consumed it (cons[p]);
//   * S3 (accumulator over the drained H0 columns) consumes h2 panels 0-3 under E2(H1) and 4-7 as they arrive;
//   * after S3 the workers first build the next tile's a1 so that S1(H1) of the next tile runs under E3.
constexpr int kBarBytes4 = 256;
constexpr int kSmemBytes4 = kARegionBytes + kStages * kStageBytes + kBiasBytes + kBarBytes4;   // 231,680 B

template <bool kBwd, bool kSaveMask, bool kF16>
__global__ void __launch_bounds__(kThreadsTC2, 1) k_nn_tc4(const TCParams prm) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  constexpr int S = kStages;
  uint8_t* sA = smem;
  uint8_t* sB = smem + kARegionBytes;
  float* sBias = reinterpret_cast<float*>(smem + kARegionBytes + S * kStageBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kARegionBytes + S * kStageBytes + kBiasBytes);
  // bars: [0,S) full  [S,2S) empty  [2S] a1_ready  [2S+1,2S+3) accfull H0/H1  [2S+3] accfree_H0  [2S+4,2S+12) panel_ready
  //       [2S+12,2S+16) cons  [2S+16] tmem slot
  const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[S]);
  const uint32_t a1_ready = smem_u32(&bars[2 * S]), accfull0 = smem_u32(&bars[2 * S + 1]);
  const uint32_t accfree_h0 = smem_u32(&bars[2 * S + 3]), panel0 = smem_u32(&bars[2 * S + 4]);
  const uint32_t cons0 = smem_u32(&bars[2 * S + 12]);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(&bars[2 * S + 16]);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < S; ++i) {
      mbar_init(full0 + 8 * i, 1);
      mbar_init(empty0 + 8 * i, 1);
    }
    mbar_init(a1_ready, 8);               // one arrival per worker warp
    mbar_init(accfull0, 1);
    mbar_init(accfull0 + 8, 1);
    mbar_init(accfree_h0, 8);
    for (int i = 0; i < 8; ++i) mbar_init(panel0 + 8 * i, 8);
    for (int i = 0; i < 4; ++i) mbar_init(cons0 + 8 * i, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_u32(tmem_slot), kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t img3_bytes = (uint32_t)prm.n3p * 128u;

  if (warp == 0) {
    // ===================== producer: weight images in the order the MMA thread consumes them =====================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      const uint8_t* w1 = reinterpret_cast<const uint8_t*>(prm.wimg);
      const uint8_t* w2 = w1 + (size_t)2 * prm.k1_panels * kStageBytes;
      const uint8_t* w3 = w2 + (size_t)2 * kNumPanels * kStageBytes;
      auto push = [&](const uint8_t* src, uint32_t bytes) {
        mbar_wait(empty0 + 8 * stage, phase ^ 1);
        mbar_expect_tx(full0 + 8 * stage, bytes);
        bulk_g2s(smem_u32(sB + stage * kStageBytes), src, bytes, full0 + 8 * stage);
        if (++stage == (uint32_t)S) { stage = 0; phase ^= 1; }
      };
      for (int round = 0; round < prm.num_rounds; ++round) {
        for (int half = 1; half >= 0; --half)                       // S1(H1) is issued before S1(H0)
          for (int kp = 0; kp < prm.k1_panels; ++kp) push(w1 + (size_t)(half * prm.k1_panels + kp) * kStageBytes, kStageBytes);
        for (int i = 0; i < 2 * kNumPanels; ++i) push(w2 + (size_t)i * kStageBytes, kStageBytes);
        for (int kp = 0; kp < kNumPanels; ++kp) push(w3 + (size_t)kp * img3_bytes, img3_bytes);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      const uint32_t a_base = smem_u32(sA);
      constexpr uint32_t idesc256 = make_idesc(256);                                   // stage 1: split-bf16 rows x bf16 weights
      // kF16 (forward only): the hidden activations and the stage-2/3 weights are fp16 (10 mantissa bits; activations
      // are O(1..100)); the backward "activations" are gradients of unbounded range and always bf16
      constexpr uint32_t idesc256h = kF16 ? make_idesc_f16(256) : make_idesc(256);
      const uint32_t idesc3 = kF16 ? make_idesc_f16(prm.n3p) : make_idesc(prm.n3p);
      // one K panel (<= 4 MMAs of K = 16): A = operand panel kp, B = the ring slot that holds the next image
      auto kblock = [&](uint32_t d_tmem, int kp, int steps, uint32_t idesc, bool first) {
        mbar_wait(full0 + 8 * stage, phase);
        tc_fence_after();
        const uint64_t da = make_desc(a_base + kp * kPanelBytes);
        const uint64_t db = make_desc(smem_u32(sB + stage * kStageBytes));
        for (int k = 0; k < steps; ++k) umma_bf16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, !(first && k == 0));
        umma_commit(empty0 + 8 * stage);
        if (++stage == (uint32_t)S) { stage = 0; phase ^= 1; }
      };
      const uint32_t h0 = tmem_base, h1 = tmem_base + 256u;
      for (int round = 0; round < prm.num_rounds; ++round) {
        mbar_wait(a1_ready, round & 1);
        tc_fence_after();
        // ---- stage 1 (conv3x3 / conv3^T on the split-bf16 im2col rows): H1 first, H0 once E3 of the previous tile has drained it
        for (int kp = 0; kp < prm.k1_panels; ++kp) kblock(h1, kp, min(4, prm.k1_steps - 4 * kp), idesc256, kp == 0);
        umma_commit(accfull0 + 8);
        if (round > 0) {
          mbar_wait(accfree_h0, (round - 1) & 1);
          tc_fence_after();
        }
        for (int kp = 0; kp < prm.k1_panels; ++kp) kblock(h0, kp, min(4, prm.k1_steps - 4 * kp), idesc256, kp == 0);
        umma_commit(accfull0);
        // ---- stage 2 (conv1x1), half 0: needs H0 drained (h1 panels 0-3 written), then follows E1 panel by panel
        for (int p = 0; p < 4; ++p) mbar_wait(panel0 + 8 * p, 0);
        tc_fence_after();
        for (int kp = 0; kp < kNumPanels; ++kp) {
          if (kp >= 4) {
            mbar_wait(panel0 + 8 * kp, 0);
            tc_fence_after();
          }
          kblock(h0, kp, 4, idesc256h, kp == 0);
        }
        umma_commit(accfull0);
        // ---- stage 2, half 1: tells E2(H0) when each of the first four h1 panels may be overwritten by h2
        for (int kp = 0; kp < kNumPanels; ++kp) {
          kblock(h1, kp, 4, idesc256h, kp == 0);
          if (kp < 4) umma_commit(cons0 + 8 * kp);
        }
        umma_commit(accfull0 + 8);
        // ---- stage 3 (small-N GEMM on h2), accumulator over the drained H0 columns
        for (int p = 0; p < 4; ++p) mbar_wait(panel0 + 8 * p, 1);
        tc_fence_after();
        for (int kp = 0; kp < kNumPanels; ++kp) {
          if (kp >= 4) {
            mbar_wait(panel0 + 8 * kp, 1);
            tc_fence_after();
          }
          kblock(h0, kp, 4, idesc3, kp == 0);
        }
        umma_commit(accfull0);
      }
    }
  } else {
    // ===================== workers: operand build + epilogues (8 warps) =====================
    const int lq = warp & 3;                            // TMEM lane quarter this warp may access
    const int ch = (warp - 2) >> 2;                     // which 32 of the 64 columns of every panel
    const int row = lq * 32 + lane;
    const int wtid = threadIdx.x - 64;                  // 0..255
    const uint32_t t_lane = tmem_base + ((uint32_t)(lq * 32) << 16);
    uint8_t* stg = sA + kARegionBytes - ((kTileM * prm.n3p * 4 + 1023) & ~1023);   // G staging rows (host checks the fit)
    const int k1_pad = prm.k1_steps * 16;
    float4 b1v = make_float4(0.f, 0.f, 0.f, 0.f), b2v = b1v;
    if constexpr (!kBwd) {
      if (wtid < kF / 4) {
        b1v = __ldg(reinterpret_cast<const float4*>(prm.bias1) + wtid);
        b2v = __ldg(reinterpret_cast<const float4*>(prm.bias2) + wtid);
        reinterpret_cast<float4*>(sBias)[wtid] = b1v;
      }
    }
    auto arrive_warp = [&](uint32_t bar) {
      __syncwarp();
      if (lane == 0) mbar_arrive(bar);
    };
    // stage-1 operand of tile `round`: two threads per row, taps 0-4 and 5-8 (+ zero padding of the K tail).
    // M < 2^31 (checked on the host), so the pixel coordinates come from 32-bit divisions.
    const int tb = ch == 0 ? 0 : 5, te = ch == 0 ? 5 : 9;
    auto row_coords = [&](int round, long long& p, bool& valid, int& h, int& w) {
      const long long tile = (long long)round * prm.tiles_per_cta_round + blockIdx.x;
      p = tile * kTileM + row;
      valid = p < prm.M;
      w = 0; h = 0;
      if (valid) {
        const uint32_t pu = (uint32_t)p, q = pu / (uint32_t)prm.W;
        w = (int)(pu - q * (uint32_t)prm.W);
        h = (int)(q % (uint32_t)prm.H);
      }
    };
    auto finish_a1 = [&]() {
      if (ch == 1)
        for (int k = 2 * 9 * prm.src_ch; k < k1_pad; k += 2)      // both bounds are even
          *reinterpret_cast<uint32_t*>(sA + a_offset(row, k)) = 0u;
      fence_proxy_async();
      arrive_warp(a1_ready);
    };
    auto build = [&](int round) {
      long long p; bool valid; int h, w;
      row_coords(round, p, valid, h, w);
      build_a1_taps<16>(sA, row, prm.src, p, valid, h, w, prm.H, prm.W, prm.src_stride, prm.src_off, prm.tap_sign, tb, te);
      finish_a1();
    };
    // <= 4 source channels: the next tile's taps are fetched into registers while this tile's stage 2 is running
    const bool prefetch_regs = prm.src_ch <= 8;
    float pre[40];
    auto prefetch_a1 = [&](int round) {
      long long p; bool valid; int h, w;
      row_coords(round, p, valid, h, w);
      switch (prm.src_ch) {
        case 1: a1_load<1>(pre, prm.src, p, valid, h, w, prm.H, prm.W, prm.src_stride, prm.src_off, prm.tap_sign, tb, te); break;
        case 2: a1_load<2>(pre, prm.src, p, valid, h, w, prm.H, prm.W, prm.src_stride, prm.src_off, prm.tap_sign, tb, te); break;
        case 8: a1_load<8>(pre, prm.src, p, valid, h, w, prm.H, prm.W, prm.src_stride, prm.src_off, prm.tap_sign, tb, te); break;
        default: a1_load<4>(pre, prm.src, p, valid, h, w, prm.H, prm.W, prm.src_stride, prm.src_off, prm.tap_sign, tb, te); break;
      }
    };
    auto store_a1 = [&]() {
      switch (prm.src_ch) {
        case 1: a1_store<1>(sA, row, pre, tb, te); break;
        case 2: a1_store<2>(sA, row, pre, tb, te); break;
        case 8: a1_store<8>(sA, row, pre, tb, te); break;
        default: a1_store<4>(sA, row, pre, tb, te); break;
      }
      finish_a1();
    };
    for (int round = 0; round < prm.num_rounds; ++round) {
      const long long tile = (long long)round * prm.tiles_per_cta_round + blockIdx.x;
      const long long p = tile * kTileM + row;
      const bool valid = p < prm.M;
      const bool stamp = prm.dbg_out != nullptr && blockIdx.x == 0 && wtid == 0;
      long long* ts = prm.dbg_out + (long long)round * 8;
      // ---- this tile's stage-1 operand rows (all MMAs of the previous tile are complete: the panels are free).  It is
      //      stored before anything else so that S1 runs while the previous tile's G rows are still leaving (one call
      //      site: the unrolled im2col code is large)
      if (prefetch_regs) {
        if (round == 0) { prefetch_a1(0); store_a1(); }       // later tiles: stored at the end of the previous iteration
      } else {
        build(round);
      }
      if (stamp) ts[0] = clock64();
      if (ch == 0) {      // pull the tile after next towards L2
        const long long pn = p + 2ll * prm.tiles_per_cta_round * kTileM;
        if (pn < prm.M) asm volatile("prefetch.global.L2 [%0];" ::"l"(prm.src + pn * prm.src_stride));
      }
      // ---- epilogues of the two hidden layers: TMEM -> (bias, relu | mask) -> fp16 / bf16 -> swizzled smem, panel by panel.
      // Only the four-panel loop is unrolled (its TMEM loads are double-buffered in registers): fully unrolled the
      // kernel grew to 160-208 KB of code and the eight worker warps thrashed the instruction cache.
#pragma unroll 1
      for (int gemm = 0; gemm < 2; ++gemm) {
        uint32_t* mask = kBwd ? (gemm == 0 ? prm.mask2 : prm.mask1) : (gemm == 0 ? prm.mask1 : prm.mask2);
        __nv_bfloat16* dump = gemm == 0 ? prm.dump1 : prm.dump2;
        // mask words of a row are stored per worker: word ch*8 + panel covers columns [64*panel + 32*ch, +32), so that
        // each thread reads / writes its 8 words as two 16-byte accesses (the layout is private to this kernel pair)
        uint32_t mkl[4] = {0u, 0u, 0u, 0u}, mkh[4] = {0u, 0u, 0u, 0u};      // panels 0-3 (H0) / 4-7 (H1)
        if constexpr (kBwd) {
          if (valid) {
            const uint4 m0 = __ldg(reinterpret_cast<const uint4*>(mask + p * (kF / 32) + ch * 8));
            const uint4 m1 = __ldg(reinterpret_cast<const uint4*>(mask + p * (kF / 32) + ch * 8) + 1);
            mkl[0] = m0.x; mkl[1] = m0.y; mkl[2] = m0.z; mkl[3] = m0.w; mkh[0] = m1.x; mkh[1] = m1.y; mkh[2] = m1.z; mkh[3] = m1.w;
          }
        }
        // the previous tile's G rows must have left the staging area (the tail of the operand panels) before any warp
        // overwrites it with h1; forward: the same barrier publishes this layer's bias vector in sBias
        if (gemm == 0 && wtid == 0) bulk_wait_read_all();
        if (!kBwd || gemm == 0) named_bar_sync(1, kWorkers2);
#pragma unroll 1
        for (int hh = 0; hh < 2; ++hh) {
          // accumulator uses per tile: H0 = S1, S2, S3 (3 per tile); H1 = S1, S2 (2 per tile)
          const uint32_t par = hh == 0 ? (uint32_t)(round + gemm) & 1u : (uint32_t)gemm;
          mbar_wait(accfull0 + 8 * hh, par);
          tc_fence_after();
          uint32_t v[2][32];
          tmem_ld32(t_lane + (uint32_t)(hh * 256 + ch * 32), v[0]);
#pragma unroll
          for (int pp = 0; pp < 4; ++pp) {
            const int pn = 4 * hh + pp;                          // K panel of the next layer's operand
            const int j = 2 * pn + ch;                           // 32-column chunk index
            tmem_ld_wait();
            if (pp + 1 < 4) tmem_ld32(t_lane + (uint32_t)(hh * 256 + (pp + 1) * 64 + ch * 32), v[(pp + 1) & 1]);
            uint32_t pk[16];
            if constexpr (!kBwd) {
              uint32_t bits = 0;
#pragma unroll
              for (int c4 = 0; c4 < 8; ++c4) {
                const float4 b4 = reinterpret_cast<const float4*>(sBias + j * 32)[c4];
                const float f0 = __uint_as_float(v[pp & 1][4 * c4 + 0]) + b4.x, f1 = __uint_as_float(v[pp & 1][4 * c4 + 1]) + b4.y;
                const float f2 = __uint_as_float(v[pp & 1][4 * c4 + 2]) + b4.z, f3 = __uint_as_float(v[pp & 1][4 * c4 + 3]) + b4.w;
                if constexpr (kSaveMask) {
                  bits |= (f0 > 0.f ? 1u : 0u) << (4 * c4) | (f1 > 0.f ? 1u : 0u) << (4 * c4 + 1) |
                          (f2 > 0.f ? 1u : 0u) << (4 * c4 + 2) | (f3 > 0.f ? 1u : 0u) << (4 * c4 + 3);
                }
                // A hidden activation above 65504 becomes +inf and surfaces as NaN (the BASIS loops count NaNs) instead of being clamped silently.
                // cvt.rn.relu.{f16x2,bf16x2}.f32: ReLU fused into the conversion
                pk[2 * c4] = kF16 ? pack_relu_f16(f0, f1) : pack_relu_bf16(f0, f1);
                pk[2 * c4 + 1] = kF16 ? pack_relu_f16(f2, f3) : pack_relu_bf16(f2, f3);
              }
              if constexpr (kSaveMask) { if (hh) mkh[pp] = bits; else mkl[pp] = bits; }
            } else {
              const uint32_t bits = hh ? mkh[pp] : mkl[pp];
#pragma unroll
              for (int c2 = 0; c2 < 16; ++c2) {
                const float f0 = ((bits >> (2 * c2)) & 1u) ? __uint_as_float(v[pp & 1][2 * c2]) : 0.f;
                const float f1 = ((bits >> (2 * c2 + 1)) & 1u) ? __uint_as_float(v[pp & 1][2 * c2 + 1]) : 0.f;
                pk[c2] = pack_bf16(f0, f1);
              }
            }
            if (dump != nullptr && valid) {      // training: the weight-gradient GEMMs take bf16 operands
#pragma unroll
              for (int c4 = 0; c4 < 4; ++c4) {
                uint32_t d[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  if constexpr (!kF16) {
                    d[q] = pk[4 * c4 + q];
                  } else {                       // fp16 activations in the operand panels: re-round to bf16
                    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&pk[4 * c4 + q]));
                    d[q] = pack_bf16(f.x, f.y);
                  }
                }
                *reinterpret_cast<uint4*>(dump + p * kF + j * 32 + c4 * 8) = make_uint4(d[0], d[1], d[2], d[3]);
              }
            }
            // h2 panel pn replaces h1 panel pn in place: S2(H1) must have consumed it (h2 panels 4-7: S2 is complete)
            if (gemm == 1 && hh == 0) mbar_wait(cons0 + 8 * pn, round & 1);
            uint8_t* base = sA + pn * kPanelBytes + row * 128;
#pragma unroll
            for (int c4 = 0; c4 < 4; ++c4)
              *reinterpret_cast<uint4*>(base + (((ch * 4 + c4) ^ (row & 7)) << 4)) =
                  make_uint4(pk[4 * c4], pk[4 * c4 + 1], pk[4 * c4 + 2], pk[4 * c4 + 3]);
            // the proxy fence is the expensive part of a hand-over: H0 panels are only needed all together, H1 panels
            // (which the next GEMM follows panel by panel) are handed over in pairs
            if (hh == 0 ? pp == 3 : (pp & 1)) {
              fence_proxy_async();
              tc_fence_before();
              __syncwarp();
              if (lane == 0) {
                if (hh == 0) {
#pragma unroll
                  for (int q = 0; q < 4; ++q) mbar_arrive(panel0 + 8 * q);
                } else {
                  mbar_arrive(panel0 + 8 * (pn - 1));
                  mbar_arrive(panel0 + 8 * pn);
                }
              }
            }
          }
          // idle until S2(H1) completes: fetch the next tile's taps
          if (gemm == 1 && hh == 0 && prefetch_regs && round + 1 < prm.num_rounds) prefetch_a1(round + 1);
        }
        if constexpr (kSaveMask) {
          if (valid) {
            uint4* mo = reinterpret_cast<uint4*>(mask + p * (kF / 32) + ch * 8);
            mo[0] = make_uint4(mkl[0], mkl[1], mkl[2], mkl[3]);
            mo[1] = make_uint4(mkh[0], mkh[1], mkh[2], mkh[3]);
          }
        }
        if constexpr (!kBwd) {                                   // swap in the other layer's bias once everyone is done
          named_bar_sync(1, kWorkers2);
          if (wtid < kF / 4) reinterpret_cast<float4*>(sBias)[wtid] = gemm == 0 ? b2v : b1v;
        }
        if (stamp) ts[1 + gemm] = clock64();
      }

      // ---- all MMAs of this tile are complete: the operand panels are free -> build the next tile's rows first,
      //      so that its stage-1 MMAs (H1 half) run while this tile's small-N accumulator is drained
      mbar_wait(accfull0, (uint32_t)(round + 2) & 1u);
      tc_fence_after();
      if (stamp) ts[3] = clock64();
      // next tile's operand rows first (registers -> panels), so that its stage-1 MMAs run while G is drained
      if (prefetch_regs && round + 1 < prm.num_rounds) store_a1();
      if (stamp) ts[4] = clock64();
      // drain the small-N accumulator: TMEM -> registers -> fp32 staging rows in the (now free) tail of the operand
      // panels -> ONE TMA bulk store of the tile's contiguous G rows.  (Direct st.global of 16 B per row costs one
      // LSU wavefront each: ~2000 cycles per tile.)  Two 16-column chunks per wait; the two warps of a lane quarter
      // alternate chunks.
      {
        // staging / global layout of one tile of G: [n3p/4 float4 columns][128 rows][4 floats] (private to this kernel and
        // the gather kernels): consecutive lanes write consecutive 16-byte words, free of bank conflicts
        uint8_t* stg_row = stg + (size_t)row * 16;
        for (int j = ch; j < prm.n3p / 16; j += 4) {
          uint32_t v[2][16];
          const bool two = j + 2 < prm.n3p / 16;
          tmem_ld16(t_lane + (uint32_t)(j * 16), v[0]);
          if (two) tmem_ld16(t_lane + (uint32_t)((j + 2) * 16), v[1]);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            if (i == 1 && !two) break;
#pragma unroll
            for (int c4 = 0; c4 < 4; ++c4)
              *reinterpret_cast<uint4*>(stg_row + (size_t)((j + 2 * i) * 4 + c4) * (kTileM * 16)) =
                  make_uint4(v[i][4 * c4], v[i][4 * c4 + 1], v[i][4 * c4 + 2], v[i][4 * c4 + 3]);
          }
        }
        tc_fence_before();
        arrive_warp(accfree_h0);                    // H0 is drained: S1(H0) of the next tile may overwrite it
        fence_proxy_async();
        named_bar_sync(2, kWorkers2);
        if (wtid == 0) {
          if (tile * kTileM < prm.M)          // whole tiles: the G buffer is sized for M rounded up to 128 rows
            bulk_s2g(prm.out + tile * kTileM * prm.n3p, smem_u32(stg), (uint32_t)(kTileM * prm.n3p * 4));
        }
      }
      if (stamp) ts[5] = clock64();
    }
    if (wtid == 0) bulk_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, kTmemCols);
}

int g_num_sms = 0;

// ---- optional per-launch timing of the tensor-core kernel (bench.py's roofline leg): a CUDA event pair
// on the launching stream around every k_nn_tc launch while profiling is on.
bool g_prof_on = false;
std::vector<TcProfToken> g_prof_recs, g_prof_pool;
double g_prof_flops = 0.0;
double g_next_flops = 0.0;   // algorithmic FLOPs of the launch being issued (set by nn_tc_forward/backward)


template <bool kBwd, bool kSaveMask, bool kF16>
void launch_tc4(const TCParams& prm, int grid, cudaStream_t s) {
  auto kern = k_nn_tc4<kBwd, kSaveMask, kF16>;
  static bool attr_set = false;
  if (!attr_set) {
    CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes4));
    attr_set = true;
  }
  const TcProfToken tok = nn_tc_prof_begin(s);
  kern<<<grid, kThreadsTC2, kSmemBytes4, s>>>(prm);
  ASEP_LAUNCH_CHECK();
  nn_tc_prof_end(tok, s, g_next_flops);
}

template <bool kBwd>
bool run_tc(TCParams prm, cudaStream_t s) {   // returns true when G was written in the tiled layout
  if (g_num_sms == 0) {
    int dev = 0;
    CUDA_CHECK(cudaGetDevice(&dev));
    CUDA_CHECK(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  {
    ASEP_CHECK(prm.k1_panels * kPanelBytes + ((kTileM * prm.n3p * 4 + 1023) & ~1023) <= kARegionBytes, ASEP_ERR_UNSUPPORTED,
               "coupling network shape outside the tcgen05 kernel (stage-1 panels %d, stage-3 columns %d)", prm.k1_panels, prm.n3p);
    ASEP_CHECK(prm.M < (1ll << 31), ASEP_ERR_UNSUPPORTED, "more than 2^31 pixels in one coupling-network launch");
    ASEP_CHECK(stage1_width_supported(prm.src_ch, kBwd), ASEP_ERR_UNSUPPORTED,
               "coupling network input width %d outside the tcgen05 kernel", prm.src_ch);
    const long long tiles = (prm.M + kTileM - 1) / kTileM;
    const int grid = (int)std::min<long long>(tiles, g_num_sms);
    prm.tiles_per_cta_round = grid;
    prm.num_rounds = (int)((tiles + grid - 1) / grid);
    static long long* dbg = nullptr;
    static const bool timing = getenv("ASEP_TC_DBG_TIMING") != nullptr;   // read once: per-phase clock64 stamps (debug aid)
    if (timing) {
      if (!dbg) CUDA_CHECK(cudaMalloc(&dbg, 8 * 4096 * sizeof(long long)));
      ASEP_CHECK(prm.num_rounds <= 4096, ASEP_ERR_BAD_ARG, "too many rounds for the timing buffer");
      prm.dbg_out = dbg;
    }
    if constexpr (kBwd) {
      launch_tc4<true, false, false>(prm, grid, s);
    } else {
      const bool save = prm.mask1 != nullptr;
      if (prm.f16) { if (save) launch_tc4<false, true, true>(prm, grid, s); else launch_tc4<false, false, true>(prm, grid, s); }
      else { if (save) launch_tc4<false, true, false>(prm, grid, s); else launch_tc4<false, false, false>(prm, grid, s); }
    }
    if (timing) {
      CUDA_CHECK(cudaStreamSynchronize(s));
      std::vector<long long> h((size_t)8 * prm.num_rounds);
      CUDA_CHECK(cudaMemcpy(h.data(), dbg, h.size() * sizeof(long long), cudaMemcpyDeviceToHost));
      double d[6] = {0};
      const int r0 = prm.num_rounds > 2 ? 1 : 0, r1 = prm.num_rounds;
      for (int r = r0; r < r1; ++r) {
        for (int i = 0; i < 5; ++i) d[i] += (double)(h[r * 8 + i + 1] - h[r * 8 + i]);
        if (r + 1 < r1) d[5] += (double)(h[(r + 1) * 8] - h[r * 8 + 5]);
      }
      const double n = r1 - r0;
      fprintf(stderr, "[tc4 %s M=%lld rounds=%d] cycles/tile: S1+E1 %.0f | E2 %.0f | wait S3 %.0f | store next a1 %.0f | E3 %.0f | gap %.0f | total %.0f\n",
              kBwd ? "bwd" : "fwd", prm.M, prm.num_rounds, d[0] / n, d[1] / n, d[2] / n, d[3] / n, d[4] / n,
              d[5] / std::max(1.0, n - 1), (double)(h[(r1 - 1) * 8 + 5] - h[r0 * 8]) / n);
      double ld = 0;
      for (int r = r0; r < r1; ++r) ld += (double)(h[r * 8 + 6] - h[r * 8 + 3]);
      fprintf(stderr, "      first E3 TMEM load complete %.0f cycles after the S3 commit was seen\n", ld / n);
    }
    return true;
  }
}

}  // namespace

TcProfToken nn_tc_prof_begin(cudaStream_t s) {
  TcProfToken rec{};
  if (!g_prof_on) return rec;
  if (!g_prof_pool.empty()) { rec = g_prof_pool.back(); g_prof_pool.pop_back(); }
  else { CUDA_CHECK(cudaEventCreate(&rec.a)); CUDA_CHECK(cudaEventCreate(&rec.b)); }
  rec.on = true;
  CUDA_CHECK(cudaEventRecord(rec.a, s));
  return rec;
}
void nn_tc_prof_end(const TcProfToken& rec, cudaStream_t s, double flops) {
  if (!rec.on) return;
  CUDA_CHECK(cudaEventRecord(rec.b, s));
  g_prof_recs.push_back(rec);
  g_prof_flops += flops;
}

void nn_tc_profile(int on) {
  g_prof_on = on != 0;
  if (g_prof_on) {
    for (auto& r : g_prof_recs) g_prof_pool.push_back(r);
    g_prof_recs.clear();
    g_prof_flops = 0.0;
  }
}
bool nn_tc_profile_enabled() { return g_prof_on; }
void nn_tc_profile_read(double* total_ms, long long* launches, double* flops) {
  double ms = 0.0;
  for (auto& r : g_prof_recs) {
    CUDA_CHECK(cudaEventSynchronize(r.b));
    float t = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&t, r.a, r.b));
    ms += t;
  }
  if (total_ms) *total_ms = ms;
  if (launches) *launches = (long long)g_prof_recs.size();
  if (flops) *flops = g_prof_flops;
}

GatherSrc nn_tc_gather_src(const NNWeightsTC& w, const NNScratchTC& sc, bool backward, long long M, int H, int W, bool split) {
  GatherSrc g;
  g.G = sc.G;
  g.const3 = backward ? nullptr : w.const3;
  g.c3 = backward ? nullptr : w.c3;
  g.n3p = backward ? w.bwd.n3p : w.fwd.n3p;
  g.H = H; g.W = W;
  g.nparts = split ? 2 : 1;
  g.part_stride = split ? (M + kTileM - 1) / kTileM * kTileM * (long long)g.n3p : 0;
  return g;
}

size_t nn_tc_g_floats(long long M, int C) { return (size_t)((M + kTileM - 1) / kTileM * kTileM) * (size_t)pad16(9 * C); }   // whole tiles

void nn_tc_prepare(NNWeightsTC& w, const float* k1, const float* c1, const float* g1, const float* b1,
                   const float* k2, const float* c2, const float* g2, const float* b2, const float* k3,
                   const float* c3, int C, int F, bool f16, bool x3) {
  ASEP_CHECK(F == kF, ASEP_ERR_UNSUPPORTED, "the tcgen05 coupling kernel is built for n_filters = %d (got %d)", kF, F);
  nn_tc_release(w);
  const int Ch = C / 2;
  // ---------------- forward
  {
    const int K1h = 9 * Ch;
    auto f1 = [&](int n, int k) { return k1[(size_t)(k % K1h) * F + n]; };              // K1[tap][ci][n]; [hi | lo]
    auto f2 = [&](int n, int k) { return g1[k] * k2[(size_t)k * F + n]; };              // diag(g1') K2
    auto f3 = [&](int n, int k) {                                                       // n = tap*C + c
      const int tap = n / C, c = n % C;
      return g2[k] * k3[((size_t)tap * F + k) * C + c];
    };
    // three-product mode with fp16 pairs: the stage-1 operand and weights are fp16 too (22 significant bits end to end)
    // The fp16 residual of an O(0.04) weight is ~1e-5, a subnormal half: the images carry 256 x w (and the kernel scales the
    // accumulators by 1/256), which keeps 22 significant bits per weight.
    const float ws = (f16 && x3) ? 256.f : 1.f;
    build_stage_set(w.fwd, 2 * K1h, 9 * C, f1, f2, f3, /*fp16 stage-2/3 weights*/ f16, /*fp16 stage 1*/ f16 && x3, false, ws);
    if (x3) build_stage_set(w.fwd_lo, 2 * K1h, 9 * C, f1, f2, f3, f16, f16, /*residual*/ true, ws);
    w.wscale_fwd = ws;
  }
  // ---------------- backward (data gradient)
  {
    const int K1h = 9 * C;
    auto f1 = [&](int n, int k) {                                                       // k = tap*C + c ; [hi | lo]
      const int kk = k % K1h, tap = kk / C, c = kk % C;
      return g2[n] * k3[((size_t)tap * F + n) * C + c];
    };
    auto f2 = [&](int n, int k) { return g1[n] * k2[(size_t)n * F + k]; };              // diag(g1') K2^T
    auto f3 = [&](int n, int k) { return k1[(size_t)n * F + k]; };                      // n = tap*Ch + ci
    build_stage_set(w.bwd, 2 * K1h, 9 * Ch, f1, f2, f3, false);
    if (x3) build_stage_set(w.bwd_lo, 2 * K1h, 9 * Ch, f1, f2, f3, false, false, /*residual*/ true);
  }
  std::vector<float> bias1(c1, c1 + F), bias2(F), const3((size_t)9 * C), vc3(c3, c3 + C);
  for (int n = 0; n < F; ++n) {
    double a = c2[n];
    for (int k = 0; k < F; ++k) a += (double)b1[k] * (double)k2[(size_t)k * F + n];
    bias2[n] = (float)a;
  }
  for (int tap = 0; tap < 9; ++tap)
    for (int c = 0; c < C; ++c) {
      double a = 0.0;
      for (int k = 0; k < F; ++k) a += (double)b2[k] * (double)k3[((size_t)tap * F + k) * C + c];
      const3[(size_t)tap * C + c] = (float)a;
    }
  w.bias1 = upload(bias1);
  w.bias2 = upload(bias2);
  w.const3 = upload(const3);
  w.c3 = upload(vc3);
  w.f16 = f16;
  w.x3 = x3;
}

void nn_tc_release(NNWeightsTC& w) {
  if (w.fwd.img) cudaFree(w.fwd.img);
  if (w.bwd.img) cudaFree(w.bwd.img);
  if (w.fwd_lo.img) cudaFree(w.fwd_lo.img);
  if (w.bwd_lo.img) cudaFree(w.bwd_lo.img);
  if (w.bias1) cudaFree(w.bias1);
  if (w.bias2) cudaFree(w.bias2);
  if (w.const3) cudaFree(w.const3);
  if (w.c3) cudaFree(w.c3);
  w = NNWeightsTC{};
}

void nn_tc_forward(const NNWeightsTC& w, const NNScratchTC& sc, const float* state, float* r, uint32_t* mask1,
                   uint32_t* mask2, int N, int H, int W, int C, cudaStream_t s, __nv_bfloat16* dump1,
                   __nv_bfloat16* dump2) {
  const long long M = (long long)N * H * W;
  if (M == 0) return;
  TCParams prm{};
  prm.src = state; prm.src_stride = C; prm.src_off = C / 2; prm.src_ch = C / 2; prm.tap_sign = 1;
  prm.wimg = w.fwd.img; prm.k1_steps = w.fwd.k1_steps; prm.k1_panels = w.fwd.k1_panels; prm.n3p = w.fwd.n3p;
  prm.bias1 = w.bias1; prm.bias2 = w.bias2; prm.mask1 = mask1; prm.mask2 = mask2;
  prm.dump1 = dump1; prm.dump2 = dump2; prm.f16 = w.f16 ? 1 : 0;
  prm.out = sc.G; prm.H = H; prm.W = W; prm.M = M;
  g_next_flops = 2.0 * (double)M * (9.0 * (C / 2) * kF + (double)kF * kF + 9.0 * kF * C);   // conv MACs x 2, unpadded
  run_tc<false>(prm, s);
  if (r != nullptr) launch_gather_fwd(sc.G, w.const3, w.c3, r, M, H, W, C, w.fwd.n3p, 1, 0, s);
}

void nn_tc_backward(const NNWeightsTC& w, const NNScratchTC& sc, const float* gr, const uint32_t* mask1,
                    const uint32_t* mask2, float* gxb, int N, int H, int W, int C, cudaStream_t s,
                    __nv_bfloat16* dump_gp2, __nv_bfloat16* dump_gp1) {
  const long long M = (long long)N * H * W;
  if (M == 0) return;
  TCParams prm{};
  prm.src = gr; prm.src_stride = C; prm.src_off = 0; prm.src_ch = C; prm.tap_sign = -1;
  prm.wimg = w.bwd.img; prm.k1_steps = w.bwd.k1_steps; prm.k1_panels = w.bwd.k1_panels; prm.n3p = w.bwd.n3p;
  prm.bias1 = nullptr; prm.bias2 = nullptr;
  prm.mask1 = const_cast<uint32_t*>(mask1); prm.mask2 = const_cast<uint32_t*>(mask2);
  prm.dump1 = dump_gp2; prm.dump2 = dump_gp1;
  prm.out = sc.G; prm.H = H; prm.W = W; prm.M = M;
  g_next_flops = 2.0 * (double)M * (9.0 * (C / 2) * kF + (double)kF * kF + 9.0 * kF * C);
  run_tc<true>(prm, s);
  if (gxb != nullptr) launch_gather_bwd(sc.G, gxb, M, H, W, C / 2, w.bwd.n3p, 1, 0, s);
}

}  // namespace asep
