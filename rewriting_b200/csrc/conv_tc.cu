// conv_tc.cu — tcgen05 implicit-GEMM over the padded-flat key layout ("row-GEMM").
//
//   acc[p, o] = sum_{tap} sum_{i} KP[p + shift(tap), i] * Wt[o, tap, i]
//
// KP is the style-modulated key  k = style (.) x  (reference: ApplyStyle,
// utils/stylegan2/models.py:616-620) stored channels-last as two bf16 planes
// (hi, lo) over a zero-padded flat pixel grid: one image = (H+1) x (W+1)
// positions, column W and row H are zero, so every 3x3 neighbour (and every
// conv_transpose phase neighbour) is a plain row shift of the same 2-D matrix
// and zero padding is implicit.  Wt is scale*W (models.py:315-319) as bf16
// hi/lo planes [Cout][tap][Cin].  Three MMAs per k-step (hi*hi + lo*hi + hi*lo)
// reproduce the fp32 conv of the reference to ~2^-17 relative (SURVEY.md §7:
// single-pass bf16/tf32 fails the 1e-3 pixel tolerance, 3xBF16 passes).
//
// Epilogue (fused, per accumulator element) follows DemodulatedConv2dF /
// NoiseInjectionF / FusedLeakyReLUF (models.py:320-328, 539-546;
// op/fused_bias_act_kernel.cu:27-47):
//   y = lrelu(acc * scale[b,o] + noise_w * noise[b, y*W+x] + bias[o], 0.2) * sqrt(2)
// each term optional, so the same kernel serves the un-fused `dconv` leaf of a
// nethook-split layer, the conv_transpose phases of an up layer and dgrad.
//
// Warp roles (192 threads): warp0 = TMA producer, warp1 = MMA issuer (+TMEM
// alloc), warps 2..5 = epilogue (TMEM -> regs -> global).  Persistent CTAs,
// 3-stage smem ring, double-buffered TMEM accumulators.
#include <cstdlib>
#include <cstring>

#include "rw_common.cuh"
#include "rw_kernels.h"

namespace rw {

namespace {

constexpr int BM = 128;
// BN (N tile = output channels per tile) is 128 for Cout % 128 == 0 and equal to Cout for the
// 64- and 32-channel tails of the 512^2 / 1024^2 generators (tcgen05 M128 takes N in steps of 16).
// BK (bf16 elements per k-block) is one swizzle row: 64 = 128 B rows (SWIZZLE_128B) in general,
// 32 = 64 B rows (SWIZZLE_64B) for Cin = 32.
constexpr int UMMA_K = 16;
constexpr int kStages = 3;
// warp 0 = TMA producer, warp 1 = MMA issuer, warps 2..9 = epilogue: two warps per TMEM lane
// quarter, each owning 64 of the tile's 128 columns (64 fp32 running sums per thread: no spills,
// and twice the epilogue throughput for the short-K phase tiles of the upsampling layers)
constexpr int kNumThreads = 320;
constexpr int kEpiWarps = 8;
// The tensor core's fp32 accumulate truncates (round-toward-zero) on every MMA: measured
// relative bias ~ -2^-25 per accumulation (profiles/r1_precision_probe.json), i.e. 1.6e-5
// after the 864 accumulations of a K=4608 tile.  So a TMEM accumulator only ever holds a
// CHUNK of kChunkKB k-blocks (K=512: 96 accumulations); the epilogue warps add the chunks in
// fp32 registers with round-to-nearest.  kNumAcc TMEM buffers form a ring between the MMA
// issuer and the epilogue.
// (kChunkKB must stay a compile-time constant: a run-time chunk bound cost 15 % in this kernel —
//  measured chunk 8 -> pixel error 5.2e-4, chunk 16 -> 8.1e-4, >= 36 fails the 1e-3 bound)
constexpr int kChunkKB = 8;
// Measured (tools/cuda/mma_rate.cu, profiles/r1_mma_rate.txt): an M=128,K=16 bf16 MMA costs
// 75 cycles for N <= 128 and 128 cycles for N = 256.  Issuing A_hi x [B_hi ; B_lo] as one N=256
// instruction (203 instead of 225 cycles per k-step) was tried and changed nothing: the kernel
// is bound by the depth of the TMA pipeline (bytes in flight vs L2 latency), not by the tensor
// pipe, so the simpler three N=128 products are kept.
template <int CG> struct AccGeom {
  static constexpr int kAccCols = 128;                     // TMEM columns per accumulator
  static constexpr int kNumAcc = 512 / kAccCols;           // ring depth
};

// CG = cta_group: 1 = one CTA per 128-row tile; 2 = CTA pair, 256-row tile, each CTA stages its
// own 128 A rows and HALF of the B (weight) tile -> 25 % less shared-memory traffic per MMA,
// which is what bounds the 1-CTA kernel (A 4 KB + B 4 KB read per 64-cycle MMA = 125 B/cycle).
template <int BN, int BK, int CG>
struct ConvSmem {
  static constexpr int kStagesN = (CG == 2) ? 4 : kStages;
  static constexpr int kABytes = BM * BK * 2;          // one plane
  static constexpr int kBBytes = (BN / CG) * BK * 2;   // one plane (this CTA's share)
  static constexpr int kStageBytes = 2 * kABytes + 2 * kBBytes;
  // per-epilogue-warp transpose scratch: 32 rows x (64 B + 16 B pad)
  static constexpr int kScratchRow = 80;
  static constexpr int kScratchBytes = kEpiWarps * 32 * kScratchRow;
  static constexpr int kTotal = kStagesN * kStageBytes + kScratchBytes + 1024 /*align slack*/ +
                                256 /*barriers*/;
};

struct Barriers {
  uint64_t full[4];
  uint64_t empty[4];
  uint64_t tmem_full[4];
  uint64_t tmem_empty[4];
  uint32_t tmem_base;
};

// tile -> (phase, mn).  Phases have very different tap counts (4/2/2/1 for a stride-2
// conv_transpose); with a static round-robin every scheduler slot would keep drawing the same
// one or two phases, so the phase is rotated by the (m, n) group index — a bijection inside
// every group of `nphase` consecutive tiles.
__device__ __forceinline__ void decode_tile(int tile, int nphase, int nsched, int& ph, int& mn) {
  mn = tile / nphase;
  ph = tile - mn * nphase;
  if (nphase > 1) ph = (ph + ((nsched % nphase) == 0 ? tile / nsched : mn)) % nphase;
}

// EPI = 0: full fused epilogue (demod, noise, bias, leaky-ReLU, NCHW / channels-last store, next
//          layer's planes, ToRGB partials — every feature a run-time switch).
// EPI = 1: lean epilogue — optional per-(b,o) scale and the store, nothing else.  The up-path
//          conv_transpose phases, dgrad and the plain row-GEMM use it: with 1-4 taps per tile the
//          mainloop is short, and the generic epilogue's ~37 predicated instructions per column
//          (2400 per tile and warp) made the MMA issuer wait for TMEM (ncu, layer 13: issuer
//          spinning on tmem_empty, tensor pipe 52 %).
//
// Every epilogue warp owns BN / 2 columns of the tile; the ToRGB partials are written per such
// column group, so a launch writes 2 * Cout / BN of them (conv_tc_rgb_parts).
template <int BN, int BK, int CG, int EPI>
__global__ void __launch_bounds__(kNumThreads, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap map_a_hi,
               const __grid_constant__ CUtensorMap map_a_lo,
               const __grid_constant__ CUtensorMap map_w_hi,
               const __grid_constant__ CUtensorMap map_w_lo, const ConvTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  using S = ConvSmem<BN, BK, CG>;
  constexpr int kSt = S::kStagesN;
  constexpr int kNumAcc = AccGeom<CG>::kNumAcc;
  constexpr int kAccCols = AccGeom<CG>::kAccCols;
  constexpr int kEpiCols = BN / 2;             // accumulator columns per epilogue warp
  constexpr int kLdCols = kEpiCols < 32 ? kEpiCols : 32;
  static_assert(BN == 128 || (CG == 1 && (BN == 64 || BN == 32)), "tile widths: 128, or 64 / 32 single-CTA");
  static_assert(BK == 64 || BK == 32, "k-block = one 128 B or 64 B swizzle row");
  static_assert(BN <= kAccCols, "accumulator does not fit its TMEM slot");
  // smem descriptors: K-major, 8-row swizzle atoms of BK * 2 bytes per row
  constexpr uint32_t kSwz = (BK == 64) ? kSwizzle128B : kSwizzle64B;
  constexpr uint32_t kSbo = 8 * BK * 2;
  uint8_t* scratch_base = smem + kSt * S::kStageBytes;
  Barriers* bars = reinterpret_cast<Barriers*>(scratch_base + S::kScratchBytes);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int cta_rank = (CG == 2) ? static_cast<int>(cluster_ctarank()) : 0;
  const bool leader = (cta_rank == 0);
  const int sched_id = blockIdx.x / CG;          // tile scheduler slot (one per CTA / CTA pair)
  const int nsched = gridDim.x / CG;

  const int m_tiles = (p.rows + BM * CG - 1) / (BM * CG);
  const int n_tiles = p.Cout / BN;
  const int mn_tiles = m_tiles * n_tiles;
  const int num_tiles = mn_tiles * p.nphase;
  const int kb_per_tap = p.Cin / BK;
  constexpr int chunk_kb = kChunkKB;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a_hi);
    tma_prefetch_desc(&map_a_lo);
    tma_prefetch_desc(&map_w_hi);
    tma_prefetch_desc(&map_w_lo);
    for (int s = 0; s < kSt; ++s) {
      mbar_init(&bars->full[s], 1);
      mbar_init(&bars->empty[s], 1);
    }
    for (int s = 0; s < kNumAcc; ++s) {
      mbar_init(&bars->tmem_full[s], 1);
      mbar_init(&bars->tmem_empty[s], kEpiWarps * CG);   // epilogue warps of every CTA of the pair
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    if constexpr (CG == 2) tmem_alloc_cg2<512>(&bars->tmem_base);
    else tmem_alloc<512>(&bars->tmem_base);
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CG == 2) cluster_sync_all();     // peer barriers are initialised
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = sched_id; tile < num_tiles; tile += nsched) {
        int ph, mn;
        decode_tile(tile, p.nphase, nsched, ph, mn);
        const int n0 = (mn % n_tiles) * BN + cta_rank * (BN / CG);
        const int m0 = (mn / n_tiles) * BM * CG + cta_rank * BM;
        for (int t = 0; t < p.ph_ntaps[ph]; ++t) {
          const int arow = m0 + p.ph_shift[ph][t];
          const int wcol = p.ph_kofs[ph][t];
          const int acol = p.ph_acol[ph][t];
          for (int kb = 0; kb < kb_per_tap; ++kb) {
            mbar_wait(&bars->empty[stage], phase ^ 1u);
            uint8_t* st = smem + stage * S::kStageBytes;
            if constexpr (CG == 2) {
              // both CTAs' bytes are credited to the leader's full barrier
              if (leader) mbar_expect_tx(&bars->full[stage], 2 * S::kStageBytes);
              tma_load_2d_cg2(st, &map_a_hi, &bars->full[stage], acol + kb * BK, arow);
              tma_load_2d_cg2(st + S::kABytes, &map_a_lo, &bars->full[stage], acol + kb * BK, arow);
              tma_load_2d_cg2(st + 2 * S::kABytes, &map_w_hi, &bars->full[stage], wcol + kb * BK, n0);
              tma_load_2d_cg2(st + 2 * S::kABytes + S::kBBytes, &map_w_lo, &bars->full[stage],
                              wcol + kb * BK, n0);
            } else {
              mbar_expect_tx(&bars->full[stage], S::kStageBytes);
              tma_load_2d(st, &map_a_hi, &bars->full[stage], acol + kb * BK, arow);
              tma_load_2d(st + S::kABytes, &map_a_lo, &bars->full[stage], acol + kb * BK, arow);
              tma_load_2d(st + 2 * S::kABytes, &map_w_hi, &bars->full[stage], wcol + kb * BK, n0);
              tma_load_2d(st + 2 * S::kABytes + S::kBBytes, &map_w_lo, &bars->full[stage],
                          wcol + kb * BK, n0);
            }
            if (++stage == kSt) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ MMA issuer --------------------------------
    constexpr uint32_t idesc = make_idesc_bf16(BM * CG, BN, 0, 0);
    int stage = 0;
    uint32_t phase = 0;
    uint32_t chunk = 0;     // running chunk counter of this CTA -> accumulator ring slot
    // All 32 lanes run this loop with warp-uniform values so that descriptors live in uniform
    // registers; one elected lane issues the tcgen05 instructions.  (Under a divergent
    // `if (lane == 0)` the compiler wraps every MMA in an ELECT / R2UR.BROADCAST waterfall loop,
    // which makes the single issuing thread the bottleneck: 12 MMAs of 75 cycles per k-block.)
    if (leader) {
      for (int tile = sched_id; tile < num_tiles; tile += nsched) {
        int ph_m, mn_m;
        decode_tile(tile, p.nphase, nsched, ph_m, mn_m);
        const int num_kb = p.ph_ntaps[ph_m] * kb_per_tap;
        for (int kb0 = 0; kb0 < num_kb; kb0 += chunk_kb, ++chunk) {
          const int as = chunk % kNumAcc;
          const uint32_t aphase = (chunk / kNumAcc) & 1u;
          mbar_wait(&bars->tmem_empty[as], aphase ^ 1u);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + as * kAccCols;
          const int kb_end = (kb0 + chunk_kb < num_kb) ? kb0 + chunk_kb : num_kb;
          for (int kb = kb0; kb < kb_end; ++kb) {
            mbar_wait(&bars->full[stage], phase);
            tc_fence_after();
            const uint32_t sa = smem_u32(smem + stage * S::kStageBytes);
            const uint64_t da_hi = make_smem_desc(sa, 16, kSbo, kSwz);
            const uint64_t da_lo = make_smem_desc(sa + S::kABytes, 16, kSbo, kSwz);
            const uint64_t db_hi = make_smem_desc(sa + 2 * S::kABytes, 16, kSbo, kSwz);
            const uint64_t db_lo = make_smem_desc(sa + 2 * S::kABytes + S::kBBytes, 16, kSbo, kSwz);
            if (elect_one()) {
#pragma unroll
              for (int kk = 0; kk < BK / UMMA_K; ++kk) {
                const uint64_t adv = static_cast<uint64_t>((kk * UMMA_K * 2) >> 4);
                // smallest terms first, then the dominant hi*hi product
                if constexpr (CG == 2) {
                  umma_bf16_cg2(tmem_d, da_lo + adv, db_hi + adv, idesc, ((kb - kb0) | kk) != 0);
                  umma_bf16_cg2(tmem_d, da_hi + adv, db_lo + adv, idesc, 1u);
                  umma_bf16_cg2(tmem_d, da_hi + adv, db_hi + adv, idesc, 1u);
                } else {
                  umma_bf16(tmem_d, da_lo + adv, db_hi + adv, idesc, ((kb - kb0) | kk) != 0);
                  umma_bf16(tmem_d, da_hi + adv, db_lo + adv, idesc, 1u);
                  umma_bf16(tmem_d, da_hi + adv, db_hi + adv, idesc, 1u);
                }
              }
              if constexpr (CG == 2) umma_commit_cg2_mc(&bars->empty[stage]);
              else umma_commit(&bars->empty[stage]);
              if (kb + 1 == kb_end) {
                if constexpr (CG == 2) umma_commit_cg2_mc(&bars->tmem_full[as]);
                else umma_commit(&bars->tmem_full[as]);
              }
            }
            __syncwarp();
            if (++stage == kSt) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else {
    // ------------------------------ epilogue ----------------------------------
    const int q = warp & 3;                 // TMEM lane quarter this warp may read
    const int half = (warp - 2) >> 2;       // which half of the tile's BN columns
    const int cbase = half * kEpiCols;
    const int img = p.Hp * p.Wp;
    uint8_t* scr = scratch_base + (warp - 2) * 32 * S::kScratchRow;
    uint32_t chunk = 0;
    for (int tile = sched_id; tile < num_tiles; tile += nsched) {
      int ph, mn;
      decode_tile(tile, p.nphase, nsched, ph, mn);
      const int num_kb = p.ph_ntaps[ph] * kb_per_tap;
      const int Hv = p.ph_Hv[ph], Wv = p.ph_Wv[ph];
      const int n0 = (mn % n_tiles) * BN + cbase;          // first output channel of this warp
      const int m0 = (mn / n_tiles) * BM * CG + cta_rank * BM;
      const int prow = m0 + q * 32 + lane;
      const int b = prow / img;
      const int rem = prow - b * img;       // prow < rows < 2^31; element offsets below are 64-bit
      const int yy = rem / p.Wp;
      const int xx = rem - yy * p.Wp;
      const bool valid = (prow < p.rows) && (yy < Hv) && (xx < Wv);

      float acc[kEpiCols];
#pragma unroll
      for (int j = 0; j < kEpiCols; ++j) acc[j] = 0.f;

      for (int kb0 = 0; kb0 < num_kb; kb0 += chunk_kb, ++chunk) {
        const int as = chunk % kNumAcc;
        const uint32_t aphase = (chunk / kNumAcc) & 1u;
        mbar_wait(&bars->tmem_full[as], aphase);
        tc_fence_after();
#pragma unroll
        for (int c0 = 0; c0 < kEpiCols; c0 += kLdCols) {
          uint32_t v[kLdCols];
          const uint32_t taddr = tmem_base + static_cast<uint32_t>(as * kAccCols + cbase + c0) +
                                 (static_cast<uint32_t>(q * 32) << 16);
          tmem_ld_32x32(taddr, v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < kLdCols; ++j) acc[c0 + j] += __uint_as_float(v[j]);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if constexpr (CG == 2) mbar_arrive_leader(&bars->tmem_empty[as]);
          else mbar_arrive(&bars->tmem_empty[as]);
        }
      }

      // ---- fused epilogue -------------------------------------------------------------
      const float* scl = p.scale_bo ? p.scale_bo + static_cast<size_t>(b) * p.Cout : nullptr;
      if constexpr (EPI == 1) {
        if (scl != nullptr && prow < p.rows) {
          const float4* s4 = reinterpret_cast<const float4*>(scl + n0);
#pragma unroll
          for (int j4 = 0; j4 < kEpiCols / 4; ++j4) {
            const float4 sv = __ldg(s4 + j4);
            acc[4 * j4] *= sv.x;
            acc[4 * j4 + 1] *= sv.y;
            acc[4 * j4 + 2] *= sv.z;
            acc[4 * j4 + 3] *= sv.w;
          }
        }
        if (p.out_mode == 0 && valid) {
          float* outp = p.out + p.ph_out_ofs[ph] + static_cast<size_t>(b) * p.out_sb +
                        static_cast<size_t>(yy) * p.out_sy + static_cast<size_t>(xx) * p.out_sx +
                        static_cast<size_t>(n0) * p.out_sc;
#pragma unroll
          for (int j = 0; j < kEpiCols; ++j) outp[static_cast<size_t>(j) * p.out_sc] = acc[j];
        }
      } else if (valid) {
        float nz = 0.f;
        if (p.noise != nullptr)
          nz = __ldg(p.noise_w) * __ldg(p.noise + static_cast<size_t>(b) * p.noise_bstride +
                                        static_cast<size_t>(yy) * Wv + xx);
        float* outp = p.out + p.ph_out_ofs[ph] + static_cast<size_t>(b) * p.out_sb +
                      static_cast<size_t>(yy) * p.out_sy + static_cast<size_t>(xx) * p.out_sx;
        const float act_gain = p.act_gain != 0.f ? p.act_gain : 1.4142135623730951f;
        const float* rw0 = p.rgb_w ? p.rgb_w + (static_cast<size_t>(b) * 3) * p.Cout : nullptr;
        float r0 = 0.f, r1 = 0.f, r2 = 0.f;
#pragma unroll
        for (int j = 0; j < kEpiCols; ++j) {
          const int o = n0 + j;
          float t = acc[j];
          if (scl) t *= __ldg(scl + o);
          t += nz;
          if (p.bias) t += __ldg(p.bias + o);
          if (p.act) t = (t > 0.f ? t : 0.2f * t) * act_gain;
          acc[j] = t;
          if (p.out != nullptr && p.out_mode == 0) outp[static_cast<size_t>(o) * p.out_sc] = t;
          if (rw0) {
            r0 = fmaf(__ldg(rw0 + o), t, r0);
            r1 = fmaf(__ldg(rw0 + p.Cout + o), t, r1);
            r2 = fmaf(__ldg(rw0 + 2 * p.Cout + o), t, r2);
          }
        }
        if (rw0) {
          // one partial per BN/2-channel group: rgb_part[(n_tile*2 + half)][b][c][y*Wv+x]
          const size_t hw = static_cast<size_t>(Hv) * Wv;
          float* rp = p.rgb_part +
                      ((static_cast<size_t>((mn % n_tiles) * 2 + half) * p.B + b) * 3) * hw +
                      static_cast<size_t>(yy) * Wv + xx;
          rp[0] = r0;
          rp[hw] = r1;
          rp[2 * hw] = r2;
        }
      } else if (p.out_mode == 1 && prow < p.rows && scl) {
        // channels-last raw rows are written for every row (pad rows are never read back)
#pragma unroll
        for (int j = 0; j < kEpiCols; ++j) acc[j] *= __ldg(scl + n0 + j);
      }
      // Row-per-lane registers -> global through a warp-private smem transpose, so that every
      // store instruction covers whole 64-byte row segments (8 rows x 64 B) instead of
      // 32 rows x 16 B.
      const int rr0 = lane >> 2;        // row within a group of 8
      const int c16 = lane & 3;         // 16-byte column slot
      if (p.out != nullptr && p.out_mode == 1) {
#pragma unroll
        for (int c0 = 0; c0 < kEpiCols; c0 += 16) {
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4)
            *reinterpret_cast<float4*>(scr + lane * S::kScratchRow + j4 * 16) = make_float4(
                acc[c0 + 4 * j4], acc[c0 + 4 * j4 + 1], acc[c0 + 4 * j4 + 2], acc[c0 + 4 * j4 + 3]);
          __syncwarp();
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            const int rr = it * 8 + rr0;
            const int grow = m0 + q * 32 + rr;
            const float4 v = *reinterpret_cast<const float4*>(scr + rr * S::kScratchRow + c16 * 16);
            if (grow < p.rows)
              *reinterpret_cast<float4*>(p.out + (static_cast<size_t>(ph) * p.rows + grow) * p.Cout +
                                         n0 + c0 + c16 * 4) = v;
          }
          __syncwarp();
        }
      }
      if (EPI == 0 && p.next_hi != nullptr) {
        // kSeg channels (2 * kSeg bytes of a row) per pass, kSlots 16-byte slots per row
        constexpr int kSeg = kEpiCols < 32 ? kEpiCols : 32;
        constexpr int kSlots = kSeg / 8;
        const int nr0 = lane / kSlots;
        const int n16 = lane % kSlots;
        const float* ns = p.next_scale + static_cast<size_t>(valid ? b : 0) * p.Cout + n0;
#pragma unroll
        for (int part = 0; part < kEpiCols / kSeg; ++part) {
#pragma unroll
          for (int plane = 0; plane < 2; ++plane) {
#pragma unroll
            for (int j8 = 0; j8 < kSlots; ++j8) {
              uint32_t w[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int j = part * kSeg + j8 * 8 + 2 * e;
                const float k0 = valid ? __ldg(ns + j) * acc[j] : 0.f;
                const float k1 = valid ? __ldg(ns + j + 1) * acc[j + 1] : 0.f;
                const __nv_bfloat162 hh = __floats2bfloat162_rn(k0, k1);
                if (plane == 0) {
                  w[e] = *reinterpret_cast<const uint32_t*>(&hh);
                } else {
                  const float2 hf = __bfloat1622float2(hh);
                  const __nv_bfloat162 ll = __floats2bfloat162_rn(k0 - hf.x, k1 - hf.y);
                  w[e] = *reinterpret_cast<const uint32_t*>(&ll);
                }
              }
              *reinterpret_cast<uint4*>(scr + lane * S::kScratchRow + j8 * 16) =
                  make_uint4(w[0], w[1], w[2], w[3]);
            }
            __syncwarp();
            __nv_bfloat16* dstp = static_cast<__nv_bfloat16*>(plane == 0 ? p.next_hi : p.next_lo);
#pragma unroll
            for (int it = 0; it < kSlots; ++it) {
              const int rr = it * (32 / kSlots) + nr0;
              const int grow = m0 + q * 32 + rr;
              const uint4 v = *reinterpret_cast<const uint4*>(scr + rr * S::kScratchRow + n16 * 16);
              if (grow < p.rows)
                *reinterpret_cast<uint4*>(dstp + static_cast<size_t>(grow) * p.Cout + n0 + part * kSeg +
                                          n16 * 8) = v;
            }
            __syncwarp();
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (CG == 2) cluster_sync_all();     // the peer may still signal our barriers / TMEM
  if (warp == 1) {
    tc_fence_after();
    if constexpr (CG == 2) tmem_dealloc_cg2<512>(tmem_base);
    else tmem_dealloc<512>(tmem_base);
  }
}

}  // namespace

template <int BN, int BK, int CG, int EPI>
static int conv_tc_launch_cg(const ConvTcParams& p, const void* a_hi, const void* a_lo,
                             const void* w_hi, const void* w_lo, int wk_total,
                             cudaStream_t stream) {
  constexpr uint32_t kSwzBytes = BK * 2;
  CUtensorMap ma_hi, ma_lo, mw_hi, mw_lo;
  int rc;
  const int a_cols = p.a_cols > 0 ? p.a_cols : p.Cin;
  if ((rc = make_tmap_2d_bf16(&ma_hi, a_hi, a_cols, p.rows, (uint64_t)a_cols * 2, BK, BM, kSwzBytes)))
    return rc;
  if ((rc = make_tmap_2d_bf16(&ma_lo, a_lo, a_cols, p.rows, (uint64_t)a_cols * 2, BK, BM, kSwzBytes)))
    return rc;
  if ((rc = make_tmap_2d_bf16(&mw_hi, w_hi, wk_total, p.Cout, (uint64_t)wk_total * 2, BK, BN / CG,
                              kSwzBytes)))
    return rc;
  if ((rc = make_tmap_2d_bf16(&mw_lo, w_lo, wk_total, p.Cout, (uint64_t)wk_total * 2, BK, BN / CG,
                              kSwzBytes)))
    return rc;

  using S = ConvSmem<BN, BK, CG>;
  static bool attr_set = false;
  if (!attr_set) {
    rc = check_cuda(cudaFuncSetAttribute(conv_tc_kernel<BN, BK, CG, EPI>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal),
                    "conv_tc smem attr");
    if (rc) return rc;
    attr_set = true;
  }
  const int m_tiles = (p.rows + BM * CG - 1) / (BM * CG);
  const int n_tiles = p.Cout / BN;
  const int num_tiles = m_tiles * n_tiles * p.nphase;
  int sched = device_sm_count() / CG;
  if (sched > num_tiles) sched = num_tiles;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(sched * CG);
  cfg.blockDim = dim3(kNumThreads);
  cfg.dynamicSmemBytes = S::kTotal;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if constexpr (CG == 1) {
    conv_tc_kernel<BN, BK, 1, EPI><<<sched, kNumThreads, S::kTotal, stream>>>(ma_hi, ma_lo, mw_hi,
                                                                             mw_lo, p);
    return check_cuda(cudaGetLastError(), "conv_tc launch");
  }
  return check_cuda(cudaLaunchKernelEx(&cfg, conv_tc_kernel<BN, BK, CG, EPI>, ma_hi, ma_lo, mw_hi, mw_lo,
                                       p),
                    "conv_tc launch");
}

// the single-CTA narrow tiles (N = 64 or 32 output channels, k-block 64 or 32 input channels)
template <int BN, int EPI>
static int conv_tc_launch_narrow(const ConvTcParams& p, const void* a_hi, const void* a_lo,
                                 const void* w_hi, const void* w_lo, int wk_total,
                                 cudaStream_t stream) {
  if (p.Cin % 64 == 0)
    return conv_tc_launch_cg<BN, 64, 1, EPI>(p, a_hi, a_lo, w_hi, w_lo, wk_total, stream);
  return conv_tc_launch_cg<BN, 32, 1, EPI>(p, a_hi, a_lo, w_hi, w_lo, wk_total, stream);
}

// N tile of a launch with Cout output channels: 128, else 64 / 32 for the narrow layers; 0 = none
int conv_tc_tile_n(int Cout) {
  if (Cout > 0 && Cout % 128 == 0) return 128;
  if (Cout == 64 || Cout == 32) return Cout;
  return 0;
}

int conv_tc_rgb_parts(int Cout) {
  const int bn = conv_tc_tile_n(Cout);
  return bn ? 2 * (Cout / bn) : 0;
}

// 0 = automatic (CTA pairs when the launch has at least one full wave of 256-row tiles),
// 1 / 2 = forced (tests, RW_CONV_CG environment variable)
static int g_conv_cg = -1;

int conv_tc_launch(const ConvTcParams& p, const void* a_hi, const void* a_lo, const void* w_hi,
                   const void* w_lo, int wk_total, cudaStream_t stream) {
  const int BN = conv_tc_tile_n(p.Cout);
  // Cin: a multiple of 64 (128 B k-blocks); 32 only for the narrow tiles (64 B k-blocks)
  const bool cin_ok = p.Cin > 0 && (p.Cin % 64 == 0 || (p.Cin == 32 && BN < 128));
  if (BN == 0 || !cin_ok || p.nphase < 1 || p.nphase > 4 || p.rows <= 0) {
    set_last_error("conv_tc: unsupported shape Cin=%d Cout=%d nphase=%d rows=%d (Cout must be a "
                   "multiple of 128 or 64 / 32, Cin a multiple of 64 or 32 with a narrow Cout)",
                   p.Cin, p.Cout, p.nphase, p.rows);
    return RW_ERR_BAD_ARG;
  }
  for (int i = 0; i < p.nphase; ++i)
    if (p.ph_ntaps[i] < 1 || p.ph_ntaps[i] > 9) {
      set_last_error("conv_tc: phase %d has %d taps", i, p.ph_ntaps[i]);
      return RW_ERR_BAD_ARG;
    }
  // lean epilogue when only the optional scale and the store are asked for
  const bool lean = !p.noise && !p.bias && !p.act && !p.rgb_w && !p.rgb_part && !p.next_hi &&
                    p.out != nullptr && (reinterpret_cast<uintptr_t>(p.scale_bo) & 15u) == 0;
  if (BN == 64) {
    if (lean) return conv_tc_launch_narrow<64, 1>(p, a_hi, a_lo, w_hi, w_lo, wk_total, stream);
    return conv_tc_launch_narrow<64, 0>(p, a_hi, a_lo, w_hi, w_lo, wk_total, stream);
  }
  if (BN == 32) {
    if (lean) return conv_tc_launch_narrow<32, 1>(p, a_hi, a_lo, w_hi, w_lo, wk_total, stream);
    return conv_tc_launch_narrow<32, 0>(p, a_hi, a_lo, w_hi, w_lo, wk_total, stream);
  }
  if (g_conv_cg < 0) {
    const char* e = getenv("RW_CONV_CG");
    g_conv_cg = e ? atoi(e) : 0;
  }
  int cg = g_conv_cg;
  if (cg != 1 && cg != 2) {
    // CTA pairs (4 stages of 48 KB, 25 % fewer bytes per MMA) for launches with at least one
    // full wave of 256-row tiles; the single-CTA kernel for the small layers
    const long long tiles256 = ((static_cast<long long>(p.rows) + 255) / 256) * (p.Cout / 128) * p.nphase;
    cg = (tiles256 >= device_sm_count() / 2) ? 2 : 1;
  }
  if (cg == 2) {
    if (lean) return conv_tc_launch_cg<128, 64, 2, 1>(p, a_hi, a_lo, w_hi, w_lo, wk_total, stream);
    return conv_tc_launch_cg<128, 64, 2, 0>(p, a_hi, a_lo, w_hi, w_lo, wk_total, stream);
  }
  if (lean) return conv_tc_launch_cg<128, 64, 1, 1>(p, a_hi, a_lo, w_hi, w_lo, wk_total, stream);
  return conv_tc_launch_cg<128, 64, 1, 0>(p, a_hi, a_lo, w_hi, w_lo, wk_total, stream);
}

}  // namespace rw
