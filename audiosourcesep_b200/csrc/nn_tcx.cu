// Split-precision ("exact") form of the fused coupling network on tcgen05 / TMEM (sm_100a).
//
// Why: inverse(forward(x)) re-evaluates ShiftAndLogScaleConvNet (flow_tfk_layers.py:73-84) on inputs that differ from
// the forward pass by fp32 round-off (flow_glow.py:187-196).  With one 16-bit word per hidden activation the network is
// piece-wise constant at 2^-9 (bf16) / 2^-12 (fp16); the flipped roundings random-walk over the 120 steps to ~1e-2 /
// ~1e-3, above the 1e-4 round-trip gate.  Here every hidden activation is carried as a (hi, lo) pair of 16-bit words
// (hi = rn(h), lo = rn(h - hi): 16 significant bits as bf16 pairs, 22 as fp16 pairs) and every hidden GEMM is two
// tcgen05 products against the SAME weight tile image, accumulated in the same fp32 TMEM columns:
//
//      p2 = [h1_hi | h1_lo] . [W2 ; W2]          (K = 2 x 512)
//
// The weight images are those of k_nn_tc4 (nn_tc.cu): nothing extra is stored and no extra weight bytes are streamed.
// This meets the round-trip gate (a deterministic, smooth-enough network), but the SCORE still carries the 16-bit
// weight rounding (measured at K = 40: ~5e-2 relative, as in the one-product mode): sqrt(flipped-ReLU fraction) plus
// 0.2 %-per-step Jacobian errors compounding over 120 steps.  The three-product mode (ASEP_PREC_FP16X3) adds the
// residual weight images w_lo = rn(w - rn(w)) and a third product hi . w_lo per GEMM, with fp16 pairs end to end in the
// forward network (22 significant bits: fp32-level pre-activations, hence fp32-level ReLU masks) and bf16 pairs in the
// data-gradient pass.
//
// What does not fit, and the schedule that follows from it.  A 128-pixel tile of (hi, lo) activations is 256 KB: more
// than shared memory (227 KB), and TMEM (512 columns) cannot hold p1 and p2 together.  So the tile is processed in two
// passes over the N halves q of the second hidden layer, and inside each pass in two K halves j of the first:
//
//   for q in {0, 1}:                                   TMEM region A = columns [0, 256), region B = [256, 512)
//     for j in {0, 1}:
//       S1(j)    A  = a1 . W1[:, half j]               stage-1 operand a1 = im2col(xb) as split-bf16 [hi | lo] (rebuilt
//                                                      from registers each time: its panels are reused for h1)
//       E1(j)    A -> bias + ReLU -> (hi, lo)          h1[:, half j]: hi in operand panels 0-3, lo in panels 4-7 (128 KB)
//       S2(q,j)  B += [hi | lo] . W2[half j, half q]   each 32 KB weight image is used by two K blocks (hi, lo)
//     E2(q)      B -> bias + ReLU -> (hi, lo)          h2[:, half q] over the same panels
//     S3(q)      A[0, n3p) = [hi | lo] . W3[half q]    small-N per-tap outputs (GEMM + col2im, see nn_tc.cu)
//     E3(q)      A -> staging -> one TMA bulk store    G part q; the gather kernel adds the two K-split parts
//
// E1 (a TMEM drain of 128 KB) and S1 (tiny) are evaluated twice; W2 is streamed exactly once per tile.  Hand-overs:
// workers -> MMA per pair of K panels (half_ready), MMA -> workers per GEMM (acc_ready, tcgen05.commit).
// The data-gradient kernel is the same schedule with the transposed images, ReLU masks instead of bias + ReLU, and bf16
// pairs (gradients have unbounded range).
#include "nn_tc_shared.cuh"

namespace asep {

namespace {

constexpr int kBarBytesX = 256;
constexpr int kSmemBytesX = kARegionBytes + kStages * kStageBytes + kBiasBytes + kBarBytesX;   // 231,680 B

__device__ __forceinline__ uint32_t pack_f16(float a, float b) {
  __half2 t = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}

// kRegs: the stage-1 taps of a tile (<= 8 source channels) are fetched once into registers and stored four times;
// otherwise (16 source channels: data gradient of the last block) the rows are rebuilt from global memory each time
template <bool kBwd, bool kSaveMask, bool kF16, bool kRegs>
__global__ void __launch_bounds__(kThreadsTC2, 1) k_nn_tcx(const TCParams prm) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  constexpr int S = kStages;
  uint8_t* sA = smem;
  uint8_t* sB = smem + kARegionBytes;
  float* sBias = reinterpret_cast<float*>(smem + kARegionBytes + S * kStageBytes);   // [0,256) bias1 half j, [256,512) bias2 half q
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kARegionBytes + S * kStageBytes + kBiasBytes);
  // bars: [0,S) full  [S,2S) empty  [2S] a1_ready  [2S+1] acc_ready  [2S+2,2S+4) half_ready  [2S+4] tmem slot
  const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[S]);
  const uint32_t a1_ready = smem_u32(&bars[2 * S]), acc_ready = smem_u32(&bars[2 * S + 1]);
  const uint32_t half0 = smem_u32(&bars[2 * S + 2]);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(&bars[2 * S + 4]);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < S; ++i) {
      mbar_init(full0 + 8 * i, 1);
      mbar_init(empty0 + 8 * i, 1);
    }
    mbar_init(a1_ready, 8);               // one arrival per worker warp
    mbar_init(acc_ready, 1);              // tcgen05.commit
    mbar_init(half0, 8);
    mbar_init(half0 + 8, 8);
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
      // three-product mode: every weight image is followed by its residual image (same layout, wimg_lo)
      const bool x3 = prm.wimg_lo != nullptr;
      const ptrdiff_t lo_off = x3 ? reinterpret_cast<const uint8_t*>(prm.wimg_lo) - w1 : 0;
      auto push = [&](const uint8_t* src, uint32_t bytes) {
        mbar_wait(empty0 + 8 * stage, phase ^ 1);
        mbar_expect_tx(full0 + 8 * stage, bytes);
        bulk_g2s(smem_u32(sB + stage * kStageBytes), src, bytes, full0 + 8 * stage);
        if (++stage == (uint32_t)S) { stage = 0; phase ^= 1; }
      };
      for (int round = 0; round < prm.num_rounds; ++round)
        for (int q = 0; q < 2; ++q) {
          for (int j = 0; j < 2; ++j) {
            for (int part = 0; part < (x3 ? 2 : 1); ++part)
              for (int kp = 0; kp < prm.k1_panels; ++kp)
                push(w1 + part * lo_off + (size_t)(j * prm.k1_panels + kp) * kStageBytes, kStageBytes);
            for (int pp = 0; pp < 4; ++pp)
              for (int part = 0; part < (x3 ? 2 : 1); ++part)
                push(w2 + part * lo_off + (size_t)(q * kNumPanels + 4 * j + pp) * kStageBytes, kStageBytes);
          }
          for (int pp = 0; pp < 4; ++pp)
            for (int part = 0; part < (x3 ? 2 : 1); ++part) push(w3 + part * lo_off + (size_t)(4 * q + pp) * img3_bytes, img3_bytes);
        }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0, n_a1 = 0, n_half = 0;
      const uint32_t a_base = smem_u32(sA);
      const bool x3 = prm.wimg_lo != nullptr;
      const uint32_t idesc1 = prm.f16_s1 ? make_idesc_f16(256) : make_idesc(256);      // split rows x 16-bit weights
      constexpr uint32_t idesc2 = kF16 ? make_idesc_f16(256) : make_idesc(256);
      const uint32_t idesc3 = kF16 ? make_idesc_f16(prm.n3p) : make_idesc(prm.n3p);
      const uint32_t rA = tmem_base, rB = tmem_base + 256u;
      // stage 1: one K panel (<= 4 MMAs of K = 16) of a1 against the next image of the ring
      auto kblock1 = [&](int kp, int steps, bool first) {
        mbar_wait(full0 + 8 * stage, phase);
        tc_fence_after();
        const uint64_t da = make_desc(a_base + kp * kPanelBytes);
        const uint64_t db = make_desc(smem_u32(sB + stage * kStageBytes));
        for (int k = 0; k < steps; ++k) umma_bf16(rA, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc1, !(first && k == 0));
        umma_commit(empty0 + 8 * stage);
        if (++stage == (uint32_t)S) { stage = 0; phase ^= 1; }
      };
      // hidden GEMMs: the hi panel pp and the lo panel 4 + pp against the SAME weight image
      auto kblock2 = [&](uint32_t d_tmem, int pp, uint32_t idesc, bool first) {
        mbar_wait(full0 + 8 * stage, phase);
        tc_fence_after();
        const uint64_t dh = make_desc(a_base + pp * kPanelBytes);
        const uint64_t dl = make_desc(a_base + (4 + pp) * kPanelBytes);
        const uint64_t db = make_desc(smem_u32(sB + stage * kStageBytes));
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16(d_tmem, dh + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, !(first && k == 0));
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16(d_tmem, dl + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, 1u);
        umma_commit(empty0 + 8 * stage);
        if (++stage == (uint32_t)S) { stage = 0; phase ^= 1; }
      };
      // three-product mode: the hi panel pp against the residual weight image (hi . w_lo; lo . w_lo is below 2^-32)
      auto kblock_res = [&](uint32_t d_tmem, int pp, uint32_t idesc) {
        mbar_wait(full0 + 8 * stage, phase);
        tc_fence_after();
        const uint64_t dh = make_desc(a_base + pp * kPanelBytes);
        const uint64_t db = make_desc(smem_u32(sB + stage * kStageBytes));
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16(d_tmem, dh + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, 1u);
        umma_commit(empty0 + 8 * stage);
        if (++stage == (uint32_t)S) { stage = 0; phase ^= 1; }
      };
      auto hidden_gemm = [&](uint32_t d_tmem, uint32_t idesc, bool first) {
        for (int hf = 0; hf < 2; ++hf) {
          mbar_wait(half0 + 8 * hf, n_half & 1u);
          tc_fence_after();
          for (int pp = 2 * hf; pp < 2 * hf + 2; ++pp) {
            kblock2(d_tmem, pp, idesc, first && pp == 0);
            if (x3) kblock_res(d_tmem, pp, idesc);
          }
        }
        ++n_half;
        umma_commit(acc_ready);
      };
      for (int round = 0; round < prm.num_rounds; ++round)
        for (int q = 0; q < 2; ++q) {
          for (int j = 0; j < 2; ++j) {
            mbar_wait(a1_ready, n_a1 & 1u);
            ++n_a1;
            tc_fence_after();
            for (int part = 0; part < (x3 ? 2 : 1); ++part)                                               // S1(j)
              for (int kp = 0; kp < prm.k1_panels; ++kp) kblock1(kp, min(4, prm.k1_steps - 4 * kp), part == 0 && kp == 0);
            umma_commit(acc_ready);
            hidden_gemm(rB, idesc2, j == 0);                                                              // S2(q, j)
          }
          hidden_gemm(rA, idesc3, true);                                                                  // S3(q)
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
    const float acc_scale = prm.acc_scale;               // 1 / (power of two folded into the weight images); exact
    uint32_t n_acc = 0;
    auto wait_acc = [&]() {
      mbar_wait(acc_ready, n_acc & 1u);
      ++n_acc;
      tc_fence_after();
    };
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
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(a1_ready);
    };
    float pre[kRegs ? 40 : 1];
    auto prefetch_a1 = [&](int round) {
      if constexpr (kRegs) {
        long long p; bool valid; int h, w;
        row_coords(round, p, valid, h, w);
        switch (prm.src_ch) {
          case 1: a1_load<1>(pre, prm.src, p, valid, h, w, prm.H, prm.W, prm.src_stride, prm.src_off, prm.tap_sign, tb, te); break;
          case 2: a1_load<2>(pre, prm.src, p, valid, h, w, prm.H, prm.W, prm.src_stride, prm.src_off, prm.tap_sign, tb, te); break;
          case 8: a1_load<8>(pre, prm.src, p, valid, h, w, prm.H, prm.W, prm.src_stride, prm.src_off, prm.tap_sign, tb, te); break;
          default: a1_load<4>(pre, prm.src, p, valid, h, w, prm.H, prm.W, prm.src_stride, prm.src_off, prm.tap_sign, tb, te); break;
        }
      }
    };
    // stage-1 operand rows of this tile: registers (or, for 16 source channels, global memory) -> split-bf16 panels
    auto put_a1 = [&](int round) {
      if constexpr (kRegs) {
        if (kF16 && prm.f16_s1) {                  // fp16 pairs (forward of the three-product mode)
          switch (prm.src_ch) {
            case 1: a1_store<1, true>(sA, row, pre, tb, te); break;
            case 2: a1_store<2, true>(sA, row, pre, tb, te); break;
            case 8: a1_store<8, true>(sA, row, pre, tb, te); break;
            default: a1_store<4, true>(sA, row, pre, tb, te); break;
          }
        } else {
          switch (prm.src_ch) {
            case 1: a1_store<1>(sA, row, pre, tb, te); break;
            case 2: a1_store<2>(sA, row, pre, tb, te); break;
            case 8: a1_store<8>(sA, row, pre, tb, te); break;
            default: a1_store<4>(sA, row, pre, tb, te); break;
          }
        }
      } else {
        long long p; bool valid; int h, w;
        row_coords(round, p, valid, h, w);
        build_a1_taps<16>(sA, row, prm.src, p, valid, h, w, prm.H, prm.W, prm.src_stride, prm.src_off, prm.tap_sign, tb, te);
      }
      finish_a1();
    };

    for (int round = 0; round < prm.num_rounds; ++round) {
      const long long tile = (long long)round * prm.tiles_per_cta_round + blockIdx.x;
      const long long p = tile * kTileM + row;
      const bool valid = p < prm.M;
      prefetch_a1(round);
#pragma unroll 1
      for (int q = 0; q < 2; ++q) {
        // three hidden-layer epilogues per pass: E1(j = 0), E1(j = 1), E2(q) -- ONE call site (the unrolled body is large)
#pragma unroll 1
        for (int e = 0; e < 3; ++e) {
          const int gemm = e == 2 ? 1 : 0;
          const int half = e == 2 ? q : e;
          const uint32_t region = gemm ? 256u : 0u;
          if (e < 2) {
            // all MMAs issued so far are complete (the last acc_ready wait): the operand panels are free
            if constexpr (!kBwd) {
              sBias[wtid] = __ldg(prm.bias1 + 256 * e + wtid);
              if (e == 0) sBias[256 + wtid] = __ldg(prm.bias2 + 256 * q + wtid);
            }
            put_a1(round);
            wait_acc();                                   // S1(j) complete
            // the previous G part must have left the staging area (tail of the operand panels) before h1 overwrites it;
            // the same barrier publishes the bias vectors
            if (wtid == 0) bulk_wait_read_all();
            named_bar_sync(1, kWorkers2);
          }
          uint32_t* mask = kBwd ? (gemm == 0 ? prm.mask2 : prm.mask1) : (gemm == 0 ? prm.mask1 : prm.mask2);
          // mask words of a row: word ch*8 + panel covers hidden columns [64*panel + 32*ch, +32) (layout of nn_tc.cu)
          uint32_t mk[4] = {0u, 0u, 0u, 0u};
          if constexpr (kBwd) {
            if (valid) {
              const uint4 m = __ldg(reinterpret_cast<const uint4*>(mask + p * (kF / 32) + ch * 8 + 4 * half));
              mk[0] = m.x; mk[1] = m.y; mk[2] = m.z; mk[3] = m.w;
            }
          }
          const float* bias = sBias + gemm * 256;
          // 16 accumulator columns at a time (two 16-byte operand chunks of hi and of lo): v[2][16] + hi[8] + lo[8] keep
          // the body inside the 168-register budget of a 320-thread block next to the prefetched stage-1 taps
          uint32_t v[2][16];
          tmem_ld16(t_lane + region + (uint32_t)(ch * 32), v[0]);
#pragma unroll
          for (int sub = 0; sub < 8; ++sub) {
            const int pp = sub >> 1, hx = sub & 1;      // K panel, 16-column half of this warp's 32 columns
            tmem_ld_wait();
            if (sub + 1 < 8) tmem_ld16(t_lane + region + (uint32_t)(((sub + 1) >> 1) * 64 + ch * 32 + ((sub + 1) & 1) * 16), v[(sub + 1) & 1]);
            uint32_t hi[8], lo[8];
            if constexpr (!kBwd) {
              uint32_t bits = 0;
#pragma unroll
              for (int c4 = 0; c4 < 4; ++c4) {
                const float4 b4 = reinterpret_cast<const float4*>(bias + pp * 64 + ch * 32 + hx * 16)[c4];
                float f[4];
                f[0] = fmaf(__uint_as_float(v[sub & 1][4 * c4 + 0]), acc_scale, b4.x); f[1] = fmaf(__uint_as_float(v[sub & 1][4 * c4 + 1]), acc_scale, b4.y);
                f[2] = fmaf(__uint_as_float(v[sub & 1][4 * c4 + 2]), acc_scale, b4.z); f[3] = fmaf(__uint_as_float(v[sub & 1][4 * c4 + 3]), acc_scale, b4.w);
                if constexpr (kSaveMask) {
                  bits |= (f[0] > 0.f ? 1u : 0u) << (4 * c4) | (f[1] > 0.f ? 1u : 0u) << (4 * c4 + 1) |
                          (f[2] > 0.f ? 1u : 0u) << (4 * c4 + 2) | (f[3] > 0.f ? 1u : 0u) << (4 * c4 + 3);
                }
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                  const float a = fmaxf(f[2 * t], 0.f), b = fmaxf(f[2 * t + 1], 0.f);
                  if constexpr (kF16) {
                    // above 65504 the pair is (inf, -inf) and surfaces as NaN (the BASIS loops count NaNs)
                    const uint32_t hp = pack_f16(a, b);
                    const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hp));
                    hi[2 * c4 + t] = hp;
                    lo[2 * c4 + t] = pack_f16(a - hf.x, b - hf.y);
                  } else {
                    const uint32_t hp = pack_bf16(a, b);
                    hi[2 * c4 + t] = hp;
                    lo[2 * c4 + t] = pack_bf16(a - __uint_as_float(hp << 16), b - __uint_as_float(hp & 0xffff0000u));
                  }
                }
              }
              if constexpr (kSaveMask) mk[pp] |= bits << (16 * hx);
            } else {
              const uint32_t bits = mk[pp] >> (16 * hx);
#pragma unroll
              for (int c2 = 0; c2 < 8; ++c2) {
                const float a = ((bits >> (2 * c2)) & 1u) ? __uint_as_float(v[sub & 1][2 * c2]) : 0.f;
                const float b = ((bits >> (2 * c2 + 1)) & 1u) ? __uint_as_float(v[sub & 1][2 * c2 + 1]) : 0.f;
                const uint32_t hp = pack_bf16(a, b);
                hi[c2] = hp;
                lo[c2] = pack_bf16(a - __uint_as_float(hp << 16), b - __uint_as_float(hp & 0xffff0000u));
              }
            }
            uint8_t* bh = sA + pp * kPanelBytes + row * 128;
            uint8_t* bl = bh + 4 * kPanelBytes;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              const int off = ((ch * 4 + hx * 2 + c) ^ (row & 7)) << 4;
              *reinterpret_cast<uint4*>(bh + off) = make_uint4(hi[4 * c], hi[4 * c + 1], hi[4 * c + 2], hi[4 * c + 3]);
              *reinterpret_cast<uint4*>(bl + off) = make_uint4(lo[4 * c], lo[4 * c + 1], lo[4 * c + 2], lo[4 * c + 3]);
            }
            if ((sub & 3) == 3) {                          // hand over a pair of K panels (hi and lo)
              fence_proxy_async();
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(half0 + 8 * (sub >> 2));
            }
          }
          if constexpr (kSaveMask) {
            if (valid && (gemm == 1 || q == 0))
              *reinterpret_cast<uint4*>(mask + p * (kF / 32) + ch * 8 + 4 * half) = make_uint4(mk[0], mk[1], mk[2], mk[3]);
          }
          wait_acc();                                     // S2(q, j) (e < 2) or S3(q) (e == 2) complete
        }
        // ---- E3(q): drain the small-N accumulator (region A) -> fp32 staging rows in the free tail of the operand panels
        //      -> ONE TMA bulk store of the tile's contiguous G rows (layout: [n3p/4 float4 columns][128 rows][4 floats])
        {
          uint8_t* stg_row = stg + (size_t)row * 16;
          for (int j = ch; j < prm.n3p / 16; j += 4) {
            uint32_t g[2][16];
            const bool two = j + 2 < prm.n3p / 16;
            tmem_ld16(t_lane + (uint32_t)(j * 16), g[0]);
            if (two) tmem_ld16(t_lane + (uint32_t)((j + 2) * 16), g[1]);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              if (i == 1 && !two) break;
#pragma unroll
              for (int c4 = 0; c4 < 4; ++c4)
                *reinterpret_cast<float4*>(stg_row + (size_t)((j + 2 * i) * 4 + c4) * (kTileM * 16)) =
                    make_float4(__uint_as_float(g[i][4 * c4]) * acc_scale, __uint_as_float(g[i][4 * c4 + 1]) * acc_scale,
                                __uint_as_float(g[i][4 * c4 + 2]) * acc_scale, __uint_as_float(g[i][4 * c4 + 3]) * acc_scale);
            }
          }
          tc_fence_before();
          fence_proxy_async();
          named_bar_sync(2, kWorkers2);
          if (wtid == 0) {
            if (tile * kTileM < prm.M)        // whole tiles: the G buffer is sized for M rounded up to 128 rows
              bulk_s2g(prm.out + (size_t)q * prm.part_stride + tile * kTileM * prm.n3p, smem_u32(stg),
                       (uint32_t)(kTileM * prm.n3p * 4));
          }
        }
      }
    }
    if (wtid == 0) bulk_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem_base, kTmemCols);
}

int g_num_sms_x = 0;

template <bool kBwd, bool kSaveMask, bool kF16, bool kRegs>
void launch_tcx(const TCParams& prm, int grid, double flops, cudaStream_t s) {
  auto kern = k_nn_tcx<kBwd, kSaveMask, kF16, kRegs>;
  static bool attr_set = false;
  if (!attr_set) {
    CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytesX));
    attr_set = true;
  }
  const TcProfToken tok = nn_tc_prof_begin(s);
  kern<<<grid, kThreadsTC2, kSmemBytesX, s>>>(prm);
  ASEP_LAUNCH_CHECK();
  nn_tc_prof_end(tok, s, flops);
}

template <bool kBwd>
void run_tcx(TCParams prm, double flops, cudaStream_t s) {
  if (g_num_sms_x == 0) {
    int dev = 0;
    CUDA_CHECK(cudaGetDevice(&dev));
    CUDA_CHECK(cudaDeviceGetAttribute(&g_num_sms_x, cudaDevAttrMultiProcessorCount, dev));
  }
  ASEP_CHECK(prm.k1_panels * kPanelBytes + ((kTileM * prm.n3p * 4 + 1023) & ~1023) <= kARegionBytes, ASEP_ERR_UNSUPPORTED,
             "coupling network shape outside the tcgen05 kernel (stage-1 panels %d, stage-3 columns %d)", prm.k1_panels, prm.n3p);
  ASEP_CHECK(prm.M < (1ll << 31), ASEP_ERR_UNSUPPORTED, "more than 2^31 pixels in one coupling-network launch");
  const long long tiles = (prm.M + kTileM - 1) / kTileM;
  const int grid = (int)std::min<long long>(tiles, g_num_sms_x);
  prm.tiles_per_cta_round = grid;
  prm.num_rounds = (int)((tiles + grid - 1) / grid);
  prm.part_stride = tiles * kTileM * (long long)prm.n3p;
  ASEP_CHECK(stage1_width_supported(prm.src_ch, kBwd), ASEP_ERR_UNSUPPORTED,
             "coupling network input width %d outside the tcgen05 kernel", prm.src_ch);
  if constexpr (kBwd) {
    if (prm.src_ch <= 8) launch_tcx<true, false, false, true>(prm, grid, flops, s);
    else launch_tcx<true, false, false, false>(prm, grid, flops, s);
  } else {
    const bool save = prm.mask1 != nullptr;
    if (prm.f16) { if (save) launch_tcx<false, true, true, true>(prm, grid, flops, s); else launch_tcx<false, false, true, true>(prm, grid, flops, s); }
    else { if (save) launch_tcx<false, true, false, true>(prm, grid, flops, s); else launch_tcx<false, false, false, true>(prm, grid, flops, s); }
  }
}

}  // namespace

size_t nn_tcx_g_floats(long long M, int C) { return 2 * nn_tc_g_floats(M, C); }

void nn_tcx_forward(const NNWeightsTC& w, const NNScratchTC& sc, const float* state, float* r, uint32_t* mask1,
                    uint32_t* mask2, int N, int H, int W, int C, cudaStream_t s) {
  const long long M = (long long)N * H * W;
  if (M == 0) return;
  TCParams prm{};
  prm.src = state; prm.src_stride = C; prm.src_off = C / 2; prm.src_ch = C / 2; prm.tap_sign = 1;
  prm.wimg = w.fwd.img; prm.k1_steps = w.fwd.k1_steps; prm.k1_panels = w.fwd.k1_panels; prm.n3p = w.fwd.n3p;
  prm.bias1 = w.bias1; prm.bias2 = w.bias2; prm.mask1 = mask1; prm.mask2 = mask2;
  prm.f16 = w.f16 ? 1 : 0;
  prm.wimg_lo = w.x3 ? w.fwd_lo.img : nullptr;
  prm.f16_s1 = (w.x3 && w.f16) ? 1 : 0;
  prm.acc_scale = 1.0f / w.wscale_fwd;
  prm.out = sc.G; prm.H = H; prm.W = W; prm.M = M;
  // algorithmic FLOPs of the network (2 x conv MACs, unpadded): the second product per GEMM is the price of the mode
  const double flops = 2.0 * (double)M * (9.0 * (C / 2) * kF + (double)kF * kF + 9.0 * kF * C);
  run_tcx<false>(prm, flops, s);
  const long long tiles = (M + kTileM - 1) / kTileM;
  if (r != nullptr) launch_gather_fwd(sc.G, w.const3, w.c3, r, M, H, W, C, w.fwd.n3p, 2, tiles * kTileM * (long long)w.fwd.n3p, s);
}

void nn_tcx_backward(const NNWeightsTC& w, const NNScratchTC& sc, const float* gr, const uint32_t* mask1,
                     const uint32_t* mask2, float* gxb, int N, int H, int W, int C, cudaStream_t s) {
  const long long M = (long long)N * H * W;
  if (M == 0) return;
  TCParams prm{};
  prm.src = gr; prm.src_stride = C; prm.src_off = 0; prm.src_ch = C; prm.tap_sign = -1;
  prm.wimg = w.bwd.img; prm.k1_steps = w.bwd.k1_steps; prm.k1_panels = w.bwd.k1_panels; prm.n3p = w.bwd.n3p;
  prm.mask1 = const_cast<uint32_t*>(mask1); prm.mask2 = const_cast<uint32_t*>(mask2);
  prm.wimg_lo = w.x3 ? w.bwd_lo.img : nullptr;
  prm.acc_scale = 1.0f;
  prm.out = sc.G; prm.H = H; prm.W = W; prm.M = M;
  const double flops = 2.0 * (double)M * (9.0 * (C / 2) * kF + (double)kF * kF + 9.0 * kF * C);
  run_tcx<true>(prm, flops, s);
  const long long tiles = (M + kTileM - 1) / kTileM;
  if (gxb != nullptr) launch_gather_bwd(sc.G, gxb, M, H, W, C / 2, w.bwd.n3p, 2, tiles * kTileM * (long long)w.bwd.n3p, s);
}

}  // namespace asep
