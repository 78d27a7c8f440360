// The whole MLP branch of Block.forward in ONE kernel (vit_models/dynamic_vit.py:159-175, :263-283; SURVEY.md section 8f
// rank 1 "fuse LN2 + MLP"), inference, bf16, D = 384:
//
//     u  = GELU(h W1^T + b1)            (B*T, 4D)   never leaves the SM
//     x' = x + bf16(u W2^T + b2)        residual stream
//     hn = LayerNorm(x') gamma + beta   input of the next block's attention (optional)
//
// Separately, fc1 + GELU writes and fc2 re-reads the (B*T, 4D) hidden tensor: 1.24 GB per layer at B = 1024, T = 197, which
// makes fc1 store-bound and is 60 % of the MLP's HBM traffic.  Here a CTA pair (tcgen05 cta_group::2, 256 rows) walks the
// hidden dimension in chunks of 128 columns:
//     G1(j): S_j (256 x 128)  = H (256 x 384, resident in shared memory)  x  W1[128 j .. 128 j + 127, :]^T     -> TMEM
//     E1(j): P_j = bf16(GELU(S_j + b1))  TMEM -> registers -> shared memory as the SWIZZLE_128B A operand of
//     G2(j): ACC (256 x 384) += P_j (256 x 128)  x  W2[:, 128 j .. 128 j + 127]^T                              -> TMEM
// (384 + 128 = 512 TMEM columns).  A tcgen05.mma fetches its 128 x 16 A slice from shared memory in ~64 cycles whatever N is, so
// N = 64 chunks ran G1 at half rate (measured: 64 cycles per MMA for 32 cycles of math); N = 128 is the break-even.  S and P are
// single-buffered: S is free once E1 holds it in registers, so the tensor pipe runs G1(j+1) and then G2(j-1)... under E1(j).  W1 / W2 chunks stream from L2 through two TMA rings (each CTA
// loads half of every weight tile).  After the last chunk a separate set of warps drains ACC: bias, round, residual add,
// LayerNorm statistics, x' and hn, while the GEMM / activation warps are already on the next row tile.
//
//   warp 0      TMA producer: H tile (once per row tile) and W1 k-blocks      warp 2   TMA producer: W2 chunks
//   warp 1      TMEM allocation; G1 issue (leader CTA only)                   warp 3   G2 issue (leader CTA only)
//   warps 4-11  E1: GELU of the hidden chunks (two groups of four warps, 64 columns each)
//   warps 12-15 output: residual add + LayerNorm of the finished row tile, overlapped with the next tile's GEMMs
// Measured alternatives, removed:
//   * 16 E1 warps (four groups of 32 columns under setmaxnreg): slower -- the stage is bound by the sub-partitions' issue / MUFU
//     slots, not by per-warp latency.
//   * The activation stage without its arithmetic: 412 -> 399 us at T = 197, i.e. the GELU is not what bounds the kernel.
// -DD2S_GEMM_TRACE_BUILD (profiling builds): clock64 totals of the issuers' barrier waits into MpParams::trace, a device buffer
// named by the D2S_GEMM_TRACE environment variable.
#include <stdlib.h>
#include "d2s_tc.cuh"

namespace d2s {

constexpr int kMpBM = 128, kMpD = 384, kMpCH = 128, kMpKB = kMpD / 64;
constexpr int kMpW1Slots = 5, kMpW2Slots = 3;   // weight ring depths
constexpr uint32_t kMpA1Blk = 128 * 128;        // 16 KB: 128 rows x 64 bf16 of H
constexpr uint32_t kMpW1Blk = 64 * 128;         //  8 KB: this CTA's 64 of the 128 W1 rows of a chunk, one k-block
constexpr uint32_t kMpW2Blk = 96 * 128;         // 12 KB: this CTA's 96 of the 192 W2 rows of one N-half, 64 of the chunk's 128 hidden columns
constexpr uint32_t kMpPBlk = 128 * 128;         // 16 KB: 128 rows x 64 bf16; P_j is two of them
constexpr int kMpE1Warps = 8, kMpOutWarps = 4, kMpThreads = (4 + kMpE1Warps + kMpOutWarps) * 32;
constexpr int kMpE1Parts = kMpE1Warps / 4;          // E1 warps per TMEM lane quadrant
constexpr int kMpE1Cols = kMpCH / kMpE1Parts;       // hidden columns of a chunk per E1 warp
constexpr uint32_t kMpAccCols = 384, kMpSCols = 128;

// clock64 totals of the issuing warps' waits (profiling builds only: D2S_NVCC_EXTRA=-DD2S_GEMM_TRACE_BUILD)
#ifdef D2S_GEMM_TRACE_BUILD
#define MP_TRACE_DECL long long tr[8] = {}; long long tr_t = clock64();
#define MP_TRACE(i) { const long long tr_n = clock64(); tr[i] += tr_n - tr_t; tr_t = tr_n; }
#define MP_TRACE_DUMP(w, n) if (p.trace && lane == 0) { long long* d_ = p.trace + ((size_t)(blockIdx.x >> 1) * 2 + (w)) * 8; \
    for (int i = 0; i < 7; ++i) d_[i] = tr[i]; d_[7] = (n); }
#else
#define MP_TRACE_DECL
#define MP_TRACE(i)
#define MP_TRACE_DUMP(w, n)
#endif

struct MpBars {
  uint64_t a1_full[kMpKB], a1_empty[kMpKB], w1_full[kMpW1Slots], w1_empty[kMpW1Slots], w2_full[kMpW2Slots], w2_empty[kMpW2Slots];
  uint64_t s_full, s_empty, p_full, p_empty, acc_full, acc_empty;
  uint64_t a1_ready[kMpKB];      // in_stats: the k-block of H has been normalised in place by both CTAs' output warps (leader's copy counts)
  uint32_t tmem_base, pad;
};
static_assert(sizeof(MpBars) % 8 == 0, "MpBars");

struct MpParams {
  long long* trace;             // profiling builds (-DD2S_GEMM_TRACE_BUILD): clock64 totals of the MMA thread's waits
  const __nv_bfloat16 *b1, *b2, *gamma, *beta, *x;
  __nv_bfloat16 *out_sum, *out_norm;
  float eps;
  int M, HID, want_ln;
  int T, ln_row0;               // LayerNorm output skips the first ln_row0 tokens of every T-token image (predictor norm over x[:, 1:])
  // LayerNorm of the INPUT applied on the fly (the producer wrote x' and per-row (mean, rstd) instead of a normalised copy):
  // map_a then covers x' itself, which is also the residual input x
  const float2* in_stats;
  const __nv_bfloat16 *in_gamma, *in_beta;
  float2* out_stats;            // per-row (mean, rstd) of x' (M) for a consumer that applies the next LayerNorm itself, or NULL
};

// One k-block of the raw residual stream, normalised in place by the calling warp (kLnIn): row r, 16-byte chunks ch0 .. ch0 + nch - 1.
// Out of line on purpose: the GELU loop that calls it once per row tile keeps its registers and its schedule.
__device__ __noinline__ void mp_normalize_block(unsigned char* hb, int r, int ch0, int nchunks, const uint32_t* gb, uint64_t sc,
                                                uint64_t sh) {
  for (int k = 0; k < nchunks; ++k) {
    const int ch = ch0 + k;
    uint4* ptr = reinterpret_cast<uint4*>(hb + sw128_off(r, ch));
    const uint4 t = *ptr;
    const uint32_t w[4] = {t.x, t.y, t.z, t.w};
    uint32_t o[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint2 g2 = *reinterpret_cast<const uint2*>(&gb[ch * 8 + 2 * q]);
      float h0, h1;
      f2_unpack(f2_fma(f2_fma(f2_pack(bf16_lo(w[q]), bf16_hi(w[q])), sc, sh), f2_pack(bf16_lo(g2.x), bf16_lo(g2.y)),
                       f2_pack(bf16_hi(g2.x), bf16_hi(g2.y))), h0, h1);
      o[q] = pack_bf16x2(h0, h1);
    }
    *ptr = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// Two-pass (mean, rstd) of one bf16 row of n elements whose fp32 sum s and one-pass mean are known: the rare statistics of a row far
// off zero.  The mean is s / n with one correction step (exact when representable: a constant row gets var = 0).  Out of line, so
// that the output warps keep their registers.
__device__ __noinline__ float2 bf16_row_stats_two_pass(const __nv_bfloat16* x, int n, float s, float mean1, float eps) {
  const float inv_n = 1.0f / (float)n;
  const float m = fmaf(fmaf(-mean1, (float)n, s), inv_n, mean1);
  const uint64_t nm = f2_bcast(-m);
  uint64_t acc0 = f2_bcast(0.f), acc1 = f2_bcast(0.f);
#pragma unroll 2
  for (int k = 0; k < n; k += 8) {
    const uint4 t = ld_cg16(x + k);
    const uint64_t d0 = f2_add(f2_pack(bf16_lo(t.x), bf16_hi(t.x)), nm), d1 = f2_add(f2_pack(bf16_lo(t.y), bf16_hi(t.y)), nm);
    const uint64_t d2 = f2_add(f2_pack(bf16_lo(t.z), bf16_hi(t.z)), nm), d3 = f2_add(f2_pack(bf16_lo(t.w), bf16_hi(t.w)), nm);
    acc0 = f2_fma(d2, d2, f2_fma(d0, d0, acc0));
    acc1 = f2_fma(d3, d3, f2_fma(d1, d1, acc1));
  }
  float a0, a1, b0, b1;
  f2_unpack(acc0, a0, a1);
  f2_unpack(acc1, b0, b1);
  return make_float2(m, rsqrtf(((a0 + a1) + (b0 + b1)) * inv_n + eps));
}

// kLnIn: the LayerNorm of the input is applied on the fly (MpParams::in_stats); a separate instantiation, so that the plain form
// compiles exactly as it did before the option existed
template <bool kLnIn>
__global__ void __cluster_dims__(2, 1, 1) __maxnreg__(128)
mlp_pair_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w1,
                const __grid_constant__ CUtensorMap map_w2, const MpParams p) {
  constexpr int TN = kMpD;
  extern __shared__ unsigned char smem_dyn[];
  const uint32_t raw = smem_u32(smem_dyn);
  const uint32_t padb = (1024u - (raw & 1023u)) & 1023u;
  unsigned char* a1_s = smem_dyn + padb;                                  // 6 x 16 KB
  unsigned char* p_s = a1_s + kMpKB * kMpA1Blk;                           // 2 x 16 KB: the two k-blocks of P_j
  unsigned char* w1_s = p_s + 2 * kMpPBlk;                                // 5 x 8 KB
  unsigned char* w2_s = w1_s + kMpW1Slots * kMpW1Blk;                     // 3 x 12 KB
  MpBars* bars = reinterpret_cast<MpBars*>(w2_s + kMpW2Slots * kMpW2Blk);
  float* b1_s = reinterpret_cast<float*>(bars + 1);                       // HID
  float* b2_s = b1_s + p.HID;                                             // 384: b2
  uint32_t* gb_s = reinterpret_cast<uint32_t*>(b2_s + TN);                // 384: (gamma, beta) as bf16 pairs
  uint32_t* gbin_s = gb_s + TN;                                           // 384: (gamma, beta) of the input LayerNorm (in_stats)
  unsigned char* out_s = reinterpret_cast<unsigned char*>(                  // 4 x 2 KB transposition buffers of the output warps
      (reinterpret_cast<uintptr_t>(gbin_s + TN) + 15) & ~(uintptr_t)15);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const int warp_u = warp_uniform(warp), rank_u = warp_uniform((int)rank);
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int pair_tiles = (p.M + 2 * kMpBM - 1) / (2 * kMpBM);
  const int nch = p.HID / kMpCH;

  if (tid == 0) {
    for (int i = 0; i < kMpKB; ++i) {
      mbar_init(smem_u32(&bars->a1_full[i]), 1);
      mbar_init(smem_u32(&bars->a1_empty[i]), 1);
      mbar_init(smem_u32(&bars->a1_ready[i]), 2 * kMpOutWarps);
    }
    for (int i = 0; i < kMpW1Slots; ++i) { mbar_init(smem_u32(&bars->w1_full[i]), 1); mbar_init(smem_u32(&bars->w1_empty[i]), 1); }
    for (int i = 0; i < kMpW2Slots; ++i) { mbar_init(smem_u32(&bars->w2_full[i]), 1); mbar_init(smem_u32(&bars->w2_empty[i]), 1); }
    mbar_init(smem_u32(&bars->s_full), 1);
    mbar_init(smem_u32(&bars->p_empty), 1);
    mbar_init(smem_u32(&bars->s_empty), 2 * kMpE1Warps);       // every E1 warp of both CTAs arrives per chunk
    mbar_init(smem_u32(&bars->p_full), 2 * kMpE1Warps);
    mbar_init(smem_u32(&bars->acc_full), 1);
    mbar_init(smem_u32(&bars->acc_empty), 2 * kMpOutWarps);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  for (int i = tid; i < p.HID; i += kMpThreads) b1_s[i] = p.b1 ? __bfloat162float(p.b1[i]) : 0.f;
  for (int i = tid; i < TN; i += kMpThreads) {
    b2_s[i] = p.b2 ? __bfloat162float(p.b2[i]) : 0.f;
    const __nv_bfloat16 gm = p.gamma ? p.gamma[i] : __float2bfloat16_rn(1.f), bt = p.beta ? p.beta[i] : __float2bfloat16_rn(0.f);
    gb_s[i] = (uint32_t)__bfloat16_as_ushort(gm) | ((uint32_t)__bfloat16_as_ushort(bt) << 16);
    if (kLnIn) gbin_s[i] = (uint32_t)__bfloat16_as_ushort(p.in_gamma[i]) | ((uint32_t)__bfloat16_as_ushort(p.in_beta[i]) << 16);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;

  if (warp_u < 4) {
  if (warp == 0) {
    if (lane == 0) {
      // ============================ TMA producer: H tile + W1 k-blocks (both CTAs) ============================
      uint32_t w1_it = 0, tile_i = 0;
      for (int pt = pair; pt < pair_tiles; pt += num_pairs, ++tile_i) {
        const int row0 = pt * 2 * kMpBM + (int)rank * kMpBM;
        if (pt + num_pairs < pair_tiles)      // next row tile's activations: pull them into L2 now, the TMA loads at the tile
          for (int kb = 0; kb < kMpKB; ++kb)  // boundary then see L2 latency instead of HBM latency
            asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];"
                         ::"l"(reinterpret_cast<uint64_t>(&map_a)), "r"(kb * 64), "r"(row0 + num_pairs * 2 * kMpBM) : "memory");
        for (int j = 0; j < nch; ++j)
          for (int kb = 0; kb < kMpKB; ++kb, ++w1_it) {
            if (j == 0) {   // the row tile's activations: resident for all chunks, refilled k-block by k-block
              mbar_wait(smem_u32(&bars->a1_empty[kb]), (tile_i & 1) ^ 1);
              const uint32_t fl = smem_u32(&bars->a1_full[kb]);
              if (kLnIn) {   // each CTA's own barrier: its E1 warps normalise the block before the pair's MMAs read it
                mbar_expect_tx(fl, kMpA1Blk);
                tma_load_2d(smem_u32(a1_s + kb * kMpA1Blk), &map_a, kb * 64, row0, fl);
              } else {
                if (rank == 0) mbar_expect_tx(fl, 2 * kMpA1Blk);
                tma_load_2d_pair(smem_u32(a1_s + kb * kMpA1Blk), &map_a, kb * 64, row0, mapa(fl, 0));
              }
            }
            const uint32_t s = w1_it % kMpW1Slots, n = w1_it / kMpW1Slots;
            mbar_wait(smem_u32(&bars->w1_empty[s]), (n & 1) ^ 1);
            const uint32_t fl = smem_u32(&bars->w1_full[s]);
            if (rank == 0) mbar_expect_tx(fl, 2 * kMpW1Blk);
            tma_load_2d_pair(smem_u32(w1_s + s * kMpW1Blk), &map_w1, kb * 64, j * kMpCH + (int)rank * (kMpCH / 2), mapa(fl, 0));
          }
      }
    }
  } else if (warp == 2) {
    if (lane == 0) {
      // ================================ TMA producer: W2 chunks (both CTAs) ================================
      uint32_t it = 0;
      for (int pt = pair; pt < pair_tiles; pt += num_pairs)
        for (int j = 0; j < nch; ++j)
          for (int q = 0; q < 4; ++q, ++it) {      // ring unit q = (k-block kb2 = q >> 1 of the chunk, N-half jn = q & 1)
            const uint32_t s = it % kMpW2Slots, n = it / kMpW2Slots;
            mbar_wait(smem_u32(&bars->w2_empty[s]), (n & 1) ^ 1);
            const uint32_t fl = smem_u32(&bars->w2_full[s]);
            if (rank == 0) mbar_expect_tx(fl, 2 * kMpW2Blk);
            tma_load_2d_pair(smem_u32(w2_s + s * kMpW2Blk), &map_w2, j * kMpCH + (q >> 1) * 64, (q & 1) * 192 + (int)rank * 96,
                             mapa(fl, 0));
          }
    }
  } else if (warp_u == 1) {
    if (rank_u == 0) {
      // ====== G1 issuer (leader): S_c = H x W1_chunk^T.  The whole warp runs the loop, one elected lane issues (see elect_one).
      // G1 and G2 have their own issuing warps: a single in-order issuer would hold back ready G2 work while it waits for an
      // S buffer (and vice versa); the tensor pipe interleaves the two instruction streams as their operands become ready. ======
      const uint32_t idesc1 = make_idesc(2 * kMpBM, kMpCH, 0);
      uint32_t w1_it = 0, c = 0, tile_i = 0;
      MP_TRACE_DECL
      for (int pt = pair; pt < pair_tiles; pt += num_pairs, ++tile_i)
        for (int j = 0; j < nch; ++j, ++c) {
          MP_TRACE(0)
          mbar_wait(smem_u32(&bars->s_empty), (c & 1) ^ 1);                  // E1 of the previous chunk has S in registers
          tc_fence_after();
          MP_TRACE(1)
          const uint32_t d = tmem + kMpAccCols;
          for (int kb = 0; kb < kMpKB; ++kb, ++w1_it) {
            if (j == 0) mbar_wait(smem_u32(kLnIn ? &bars->a1_ready[kb] : &bars->a1_full[kb]), tile_i & 1);
            MP_TRACE(2)
            const uint32_t s = w1_it % kMpW1Slots, n = w1_it / kMpW1Slots;
            mbar_wait(smem_u32(&bars->w1_full[s]), n & 1);
            tc_fence_after();
            MP_TRACE(3)
            const uint64_t ad = make_desc_sw128(smem_u32(a1_s + kb * kMpA1Blk), 16, 1024);
            const uint64_t bd = make_desc_sw128(smem_u32(w1_s + s * kMpW1Blk), 16, 1024);
            if (elect_one()) {
              if (kb == 0) mma2_ss_imm<false>(d, ad, bd, idesc1); else mma2_ss_imm<true>(d, ad, bd, idesc1);
              mma2_ss_imm<true>(d, ad + 2, bd + 2, idesc1);
              mma2_ss_imm<true>(d, ad + 4, bd + 4, idesc1);
              mma2_ss_imm<true>(d, ad + 6, bd + 6, idesc1);
              mma2_commit_both(smem_u32(&bars->w1_empty[s]));
              if (j == nch - 1) mma2_commit_both(smem_u32(&bars->a1_empty[kb]));   // last reader of this H k-block
            }
            __syncwarp();
          }
          if (elect_one()) mma2_commit_both(smem_u32(&bars->s_full));
          __syncwarp();
        }
      MP_TRACE(0)
      MP_TRACE_DUMP(0, c)
    }
  } else if (warp_u == 3) {
    if (rank_u == 0) {
      // ====== G2 issuer (leader): ACC += P_c x W2_chunk^T ======
      const uint32_t idesc2 = make_idesc(2 * kMpBM, 192, 0);
      uint32_t c = 0, w2_it = 0, tile_i = 0;
      MP_TRACE_DECL
      for (int pt = pair; pt < pair_tiles; pt += num_pairs, ++tile_i)
        for (int j = 0; j < nch; ++j, ++c) {
          MP_TRACE(0)
          mbar_wait(smem_u32(&bars->p_full), c & 1);                           // both CTAs' E1 warps have written P_c
          MP_TRACE(4)
          if (j == 0) mbar_wait(smem_u32(&bars->acc_empty), (tile_i & 1) ^ 1);   // previous tile's output warps have drained ACC
          tc_fence_after();
          MP_TRACE(6)
#pragma unroll
          for (int q = 0; q < 4; ++q, ++w2_it) {     // (k-block kb2 = q >> 1 of P_c, N-half jn = q & 1)
            const uint32_t s = w2_it % kMpW2Slots, n = w2_it / kMpW2Slots;
            mbar_wait(smem_u32(&bars->w2_full[s]), n & 1);
            tc_fence_after();
            MP_TRACE(5)
            const uint64_t ad = make_desc_sw128(smem_u32(p_s + (q >> 1) * kMpPBlk), 16, 1024);
            const uint64_t bd = make_desc_sw128(smem_u32(w2_s + s * kMpW2Blk), 16, 1024);
            const uint32_t d = tmem + (q & 1) * 192;
            if (elect_one()) {
              if (j == 0 && q < 2) mma2_ss_imm<false>(d, ad, bd, idesc2); else mma2_ss_imm<true>(d, ad, bd, idesc2);
              mma2_ss_imm<true>(d, ad + 2, bd + 2, idesc2);
              mma2_ss_imm<true>(d, ad + 4, bd + 4, idesc2);
              mma2_ss_imm<true>(d, ad + 6, bd + 6, idesc2);
              mma2_commit_both(smem_u32(&bars->w2_empty[s]));
              if (q == 3) {
                mma2_commit_both(smem_u32(&bars->p_empty));
                if (j == nch - 1) mma2_commit_both(smem_u32(&bars->acc_full));
              }
            }
            __syncwarp();
          }
        }
      MP_TRACE(0)
      MP_TRACE_DUMP(1, c)
    }
  }
  } else if (warp_u < 4 + kMpE1Warps) {
    // ============================== E1 warps (both CTAs): P_j = bf16(GELU(S_j + b1)) ==============================
    // Two warps per TMEM lane quadrant, 64 of the chunk's 128 columns each (= one of the two k-blocks of P_j).  S and P are
    // single-buffered: S is free again as soon as it sits in registers (G1 of the next chunk then runs under this chunk's
    // GELU), P as soon as G2 of the previous chunk has retired (which the tensor pipe executes under this chunk's GELU too).
    const int ew = warp - 4;                    // 0 .. kMpE1Warps-1
    const int quad = warp & 3;                  // TMEM lane quadrant of this warp
    const int part = ew >> 2;                   // which kMpE1Cols of the chunk's 128 columns
    const int r = quad * 32 + lane;
    const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16) + kMpAccCols + part * kMpE1Cols;
    // P_j is two SWIZZLE_128B k-blocks of 64 columns; this warp's columns are 16-byte chunks kc0 .. of block pblk
    unsigned char* blk = p_s + (part * kMpE1Cols / 64) * kMpPBlk;
    const int kc0 = (part * kMpE1Cols % 64) / 8;
    uint32_t c = 0;
    for (int pt = pair; pt < pair_tiles; pt += num_pairs)
      for (int j = 0; j < nch; ++j, ++c) {
        mbar_wait(smem_u32(&bars->s_full), c & 1);
        tc_fence_after();
        // all columns first: S_j is then in registers and G1(j + 1) may overwrite it while the GELU below runs (with the
        // second half loaded after the first half's GELU, s_empty went out ~1 k cycles later and G1 waited for it)
        uint32_t va[32], vb[32];
        tmem_ld32_nowait(lane_addr, va);
        if (kMpE1Cols == 64) tmem_ld32_nowait(lane_addr + 32, vb);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(mapa(smem_u32(&bars->s_empty), 0));
        uint32_t o[kMpE1Cols / 2];
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          const float2 bq = *reinterpret_cast<const float2*>(&b1_s[j * kMpCH + part * kMpE1Cols + 2 * q]);
          float g0, g1;
          f2_unpack(gelu_erf_pair(f2_add(f2_pack(__uint_as_float(va[2 * q]), __uint_as_float(va[2 * q + 1])), f2_pack(bq.x, bq.y))), g0, g1);
          o[q] = pack_bf16x2(g0, g1);
        }
        if (kMpE1Cols == 64) {
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            const float2 bq = *reinterpret_cast<const float2*>(&b1_s[j * kMpCH + part * kMpE1Cols + 32 + 2 * q]);
            float g0, g1;
            f2_unpack(gelu_erf_pair(f2_add(f2_pack(__uint_as_float(vb[2 * q]), __uint_as_float(vb[2 * q + 1])), f2_pack(bq.x, bq.y))), g0, g1);
            o[(kMpE1Cols == 64 ? 16 : 0) + q] = pack_bf16x2(g0, g1);
          }
        }
        mbar_wait(smem_u32(&bars->p_empty), (c & 1) ^ 1);                             // G2(j - 1) has read P
#pragma unroll
        for (int k = 0; k < kMpE1Cols / 8; ++k)
          *reinterpret_cast<uint4*>(blk + sw128_off(r, kc0 + k)) = make_uint4(o[4 * k], o[4 * k + 1], o[4 * k + 2], o[4 * k + 3]);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");                  // generic-proxy writes -> visible to the MMA
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(mapa(smem_u32(&bars->p_full), 0));
      }
  } else {
    // ===================== output warps (both CTAs): x' = x + bf16(ACC + b2), hn = LayerNorm(x') =====================
    // Their own 4 warps (one per TMEM lane quadrant; a thread owns one row, all 384 columns), so a tile's residual add,
    // LayerNorm and ~300 KB of loads / stores run under the NEXT tile's GEMMs (with the E1 warps doing this too, a third of
    // every tile was spent here with the tensor pipe idle).  Global memory is touched in coalesced 64-byte row segments
    // through a 2 KB per-warp transposition buffer.  x' is not kept in registers: pass 2 re-reads it (L2-hot) once the row's
    // mean and variance are known.  Only pass 1 holds the accumulator, so G2 of the next tile waits for little.
    const int quad = warp & 3;
    const int ow = warp - 4 - kMpE1Warps;       // 0..3
    const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16);
    unsigned char* buf = out_s + ow * 2048;                     // [32 rows x 64 B]
    const int crow = lane >> 2, cseg = lane & 3;                // coalesced pattern: 4 lanes x 16 B cover one row's 64 bytes
    const uint32_t own_off = (uint32_t)lane * 64, own_sw = (uint32_t)(lane >> 1) & 3u;
    constexpr int NU = TN / 32;                                  // 32-column units per row
    // kLnIn: H arrives as the raw residual stream x'; the output warps normalise it in place, one row per thread, h = bf16(((x -
    // mean) * rstd) * gamma + beta) with the producer's statistics -- the arithmetic of the pair GEMM's own LayerNorm pass, so the
    // A operand is bit-identical to the normalised copy that is no longer written.  The NEXT row tile's blocks land when G1 of
    // the current tile's last chunk has retired, i.e. while these warps are waiting for the current accumulator anyway: G1(0) of
    // the next tile still starts under the current tile's last GELU, and the GELU warps (the kernel's critical stage) do not
    // see any of it.
    auto normalize_tile = [&](int pt_n, uint32_t ti) {
      const int r = quad * 32 + lane;
      const int row = pt_n * 2 * kMpBM + (int)rank * kMpBM + r;
      const float2 st = row < p.M ? p.in_stats[row] : make_float2(0.f, 0.f);
      const uint64_t sc = f2_bcast(st.y), sh = f2_bcast(-st.x * st.y);
#pragma unroll 1
      for (int kb = 0; kb < kMpKB; ++kb) {
        mbar_wait(smem_u32(&bars->a1_full[kb]), ti & 1);
        mp_normalize_block(a1_s + kb * kMpA1Blk, r, 0, 8, gbin_s + kb * 64, sc, sh);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(mapa(smem_u32(&bars->a1_ready[kb]), 0));
      }
    };
    uint32_t tile_i = 0;
    if (kLnIn && pair < pair_tiles) normalize_tile(pair, 0);
    for (int pt = pair; pt < pair_tiles; pt += num_pairs, ++tile_i) {
      if (kLnIn && pt + num_pairs < pair_tiles) normalize_tile(pt + num_pairs, tile_i + 1);
      const int row0 = pt * 2 * kMpBM + (int)rank * kMpBM + quad * 32;     // first row of this warp
      const int rows_left = p.M - row0 - crow;                             // row group i is in range iff 8 i < rows_left
      // element offsets of (row0 + crow + 8 i, cseg * 8); rows past M re-read the last row and are never stored
      size_t goff[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) goff[i] = (size_t)min(row0 + crow + 8 * i, p.M - 1) * TN + cseg * 8;
      // while the tile's GEMMs run: pull this warp's 32 residual rows (32 x 768 B = 192 lines) into L2, so that pass 1, which
      // holds the accumulator, streams them at L2 latency; and have the first unit in registers before the wait
      {
        const int prow = min(row0 + lane, p.M - 1);
#pragma unroll
        for (int k = 0; k < 6; ++k) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.x + (size_t)prow * TN + k * 64));
      }
      uint4 xn[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) xn[i] = ld_nc16(p.x + goff[i]);
      mbar_wait(smem_u32(&bars->acc_full), tile_i & 1);      // all G2 of this tile retired: ACC complete
      tc_fence_after();
      // ---- pass 1: x' = bf16(x + bf16(ACC + b2)) -> global; fp32 sum / sum of squares of the rounded values ----
      uint64_t acc_s = f2_bcast(0.f), acc_q = f2_bcast(0.f);
#pragma unroll 1
      for (int u = 0; u < NU; ++u) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int row = 8 * i + crow;
          *reinterpret_cast<uint4*>(buf + row * 64 + ((cseg ^ ((row >> 1) & 3)) << 4)) = xn[i];
        }
        if (u + 1 < NU) {
#pragma unroll
          for (int i = 0; i < 4; ++i) xn[i] = ld_nc16(p.x + goff[i] + (u + 1) * 32);       // next unit in flight
        }
        uint32_t v[32];
        tmem_ld32_nowait(lane_addr + u * 32, v);
        __syncwarp();
        uint32_t xw[16];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint4 t = *reinterpret_cast<const uint4*>(buf + own_off + (((uint32_t)q ^ own_sw) << 4));
          xw[4 * q] = t.x; xw[4 * q + 1] = t.y; xw[4 * q + 2] = t.z; xw[4 * q + 3] = t.w;
        }
        tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 16; ++q) {
          const float2 bq = *reinterpret_cast<const float2*>(&b2_s[u * 32 + 2 * q]);
          float y0, y1;
          f2_unpack(f2_add(f2_pack(__uint_as_float(v[2 * q]), __uint_as_float(v[2 * q + 1])), f2_pack(bq.x, bq.y)), y0, y1);
          const uint32_t yb = pack_bf16x2(y0, y1);                    // fc2's bf16 output
          const uint32_t sb2 = add_bf16x2(xw[q], yb);                 // the residual add's bf16 output (rounded once)
          xw[q] = sb2;
          const uint64_t sv = f2_pack(bf16_lo(sb2), bf16_hi(sb2));
          acc_s = f2_add(acc_s, sv);
          acc_q = f2_fma(sv, sv, acc_q);
        }
        __syncwarp();     // every lane has read its x row: the buffer can take x'
#pragma unroll
        for (int q = 0; q < 4; ++q)
          *reinterpret_cast<uint4*>(buf + own_off + (((uint32_t)q ^ own_sw) << 4)) = make_uint4(xw[4 * q], xw[4 * q + 1], xw[4 * q + 2], xw[4 * q + 3]);
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int row = 8 * i + crow;
          const uint4 val = *reinterpret_cast<const uint4*>(buf + row * 64 + ((cseg ^ ((row >> 1) & 3)) << 4));
          if (8 * i < rows_left) *reinterpret_cast<uint4*>(p.out_sum + goff[i] + u * 32) = val;
        }
        __syncwarp();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(mapa(smem_u32(&bars->acc_empty), 0));     // the next tile's G2(0) may start
      if (p.want_ln || p.out_stats != nullptr) {
        float s0, s1, q0, q1;
        f2_unpack(acc_s, s0, s1);
        f2_unpack(acc_q, q0, q1);
        float mean = (s0 + s1) * (1.0f / TN);
        const float var = fmaxf((q0 + q1) * (1.0f / TN) - mean * mean, 0.f);
        float rstd = rsqrtf(var + p.eps);
        // E[x^2] - mean^2 is exact enough while 8 mean^2 <= var (the sum of squares is then at most 1.125 x the squared
        // deviations).  A row farther off zero would lose log2(1 + mean^2 / var) bits to the cancellation: it gets two-pass
        // statistics instead, from the x' row this warp has just written (L2-hot; the thread re-reads its own row).
        if (row0 + lane < p.M && 8.f * mean * mean > var) {
          const float2 st = bf16_row_stats_two_pass(p.out_sum + (size_t)(row0 + lane) * TN, TN, s0 + s1, mean, p.eps);
          mean = st.x;
          rstd = st.y;
        }
        if (p.out_stats != nullptr && row0 + lane < p.M) p.out_stats[row0 + lane] = make_float2(mean, rstd);   // (this thread's row)
        if (!p.want_ln) continue;
        const uint64_t sc = f2_bcast(rstd), sh = f2_bcast(-mean * rstd);
        // ---- pass 2: hn = (x' - mean) * rstd * gamma + beta; x' comes back from L2 (this warp wrote it above) ----
        // hn row of global row g = (image b, token t): b * (T - ln_row0) + t - ln_row0, tokens t < ln_row0 are not written
        size_t hoff[4];
        bool hok[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int g = row0 + crow + 8 * i;
          const int bimg = g / p.T, t = g - bimg * p.T;
          hok[i] = 8 * i < rows_left && t >= p.ln_row0;
          hoff[i] = ((size_t)bimg * (p.T - p.ln_row0) + (size_t)max(t - p.ln_row0, 0)) * TN + cseg * 8;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) xn[i] = ld_cg16(p.out_sum + goff[i]);
#pragma unroll 1
        for (int u = 0; u < NU; ++u) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int row = 8 * i + crow;
            *reinterpret_cast<uint4*>(buf + row * 64 + ((cseg ^ ((row >> 1) & 3)) << 4)) = xn[i];
          }
          if (u + 1 < NU) {
#pragma unroll
            for (int i = 0; i < 4; ++i) xn[i] = ld_cg16(p.out_sum + goff[i] + (u + 1) * 32);
          }
          __syncwarp();
          uint32_t hw[16];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint4 t = *reinterpret_cast<const uint4*>(buf + own_off + (((uint32_t)q ^ own_sw) << 4));
            hw[4 * q] = t.x; hw[4 * q + 1] = t.y; hw[4 * q + 2] = t.z; hw[4 * q + 3] = t.w;
          }
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            const uint2 gb = *reinterpret_cast<const uint2*>(&gb_s[u * 32 + 2 * q]);     // (gamma, beta) of two columns
            float h0, h1;
            f2_unpack(f2_fma(f2_fma(f2_pack(bf16_lo(hw[q]), bf16_hi(hw[q])), sc, sh), f2_pack(bf16_lo(gb.x), bf16_lo(gb.y)),
                             f2_pack(bf16_hi(gb.x), bf16_hi(gb.y))), h0, h1);
            hw[q] = pack_bf16x2(h0, h1);
          }
          __syncwarp();
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(buf + own_off + (((uint32_t)q ^ own_sw) << 4)) = make_uint4(hw[4 * q], hw[4 * q + 1], hw[4 * q + 2], hw[4 * q + 3]);
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int row = 8 * i + crow;
            const uint4 val = *reinterpret_cast<const uint4*>(buf + row * 64 + ((cseg ^ ((row >> 1) & 3)) << 4));
            if (hok[i]) *reinterpret_cast<uint4*>(p.out_norm + hoff[i] + u * 32) = val;
          }
          __syncwarp();
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();            // the peer may still signal barriers / read operands in this CTA's shared memory
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512) : "memory");
  }
}

static int mp_map_2d(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint32_t box_inner, uint32_t box_outer,
                     CUtensorMapL2promotion promo, const char* what) {
  GgEncodeFn enc = gg_encode_fn();
  D2S_REQUIRE(enc != nullptr, D2S_ERR_CUDA, "%s: cuTensorMapEncodeTiled is unavailable from the driver", what);
  const cuuint64_t gdim[2] = {inner, outer};
  const cuuint64_t gstr[1] = {inner * 2};
  const cuuint32_t box[2] = {box_inner, box_outer};
  const cuuint32_t estr[2] = {1, 1};
  CUresult cr = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  D2S_REQUIRE(cr == CUDA_SUCCESS, D2S_ERR_CUDA, "%s: tensor map encode failed (%d)", what, (int)cr);
  return D2S_OK;
}

}  // namespace d2s

using namespace d2s;

static_assert(kMpW1Slots >= kMpKB - 1, "in_stats: the H blocks of a tile are issued interleaved with the first chunk's W1 blocks");

static int mp_launch(const char* what, const void* h, const float* in_stats, const void* in_gamma, const void* in_beta, const void* w1,
                     const void* b1, const void* w2, const void* b2, const void* x, const void* gamma, const void* beta, float eps,
                     int M, int D, int HID, int T, int norm_row0, void* out_sum, void* out_norm, float* out_stats, d2s_stream_t stream) {
  D2S_REQUIRE(h && w1 && w2 && x && out_sum, D2S_ERR_ARG, "mlp_residual_ln: null pointer");
  D2S_REQUIRE(M >= 0 && D == kMpD && HID >= kMpCH && HID % kMpCH == 0 && HID <= 2048, D2S_ERR_ARG,
              "mlp_residual_ln: need D == %d and HID %% %d == 0, %d <= HID <= 2048 (got M=%d D=%d HID=%d)", kMpD, kMpCH, kMpCH, M,
              D, HID);
  D2S_REQUIRE(!out_norm || (gamma && beta), D2S_ERR_ARG, "mlp_residual_ln: out_norm needs gamma and beta");
  D2S_REQUIRE(T >= 1 && norm_row0 >= 0 && norm_row0 < T && (norm_row0 == 0 || M % T == 0), D2S_ERR_ARG,
              "mlp_residual_ln: need 0 <= norm_row0 < T and M %% T == 0 (got M=%d T=%d norm_row0=%d)", M, T, norm_row0);
  D2S_REQUIRE(aligned16(h) && aligned16(w1) && aligned16(w2) && aligned16(x) && aligned16(out_sum) && aligned16(out_norm),
              D2S_ERR_ALIGN, "mlp_residual_ln: pointers must be 16-byte aligned");
  if (M == 0) return D2S_OK;
  CUtensorMap ma, mw1, mw2;
  int rc;
  if ((rc = mp_map_2d(&ma, h, D, M, 64, kMpBM, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, what))) return rc;
  if ((rc = mp_map_2d(&mw1, w1, D, HID, 64, kMpCH / 2, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, what))) return rc;
  if ((rc = mp_map_2d(&mw2, w2, HID, D, 64, 96, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, what))) return rc;
  const char* tr_env = getenv("D2S_GEMM_TRACE");
  MpParams p{tr_env ? reinterpret_cast<long long*>(strtoull(tr_env, nullptr, 10)) : nullptr, (const __nv_bfloat16*)b1, (const __nv_bfloat16*)b2, (const __nv_bfloat16*)gamma, (const __nv_bfloat16*)beta,
             (const __nv_bfloat16*)x, (__nv_bfloat16*)out_sum, (__nv_bfloat16*)out_norm, eps, M, HID, out_norm ? 1 : 0, T, norm_row0,
             reinterpret_cast<const float2*>(in_stats), (const __nv_bfloat16*)in_gamma, (const __nv_bfloat16*)in_beta,
             reinterpret_cast<float2*>(out_stats)};
  const size_t smem = 1024 + (size_t)kMpKB * kMpA1Blk + 2 * (size_t)kMpPBlk + (size_t)kMpW1Slots * kMpW1Blk +
                      (size_t)kMpW2Slots * kMpW2Blk + sizeof(MpBars) + (size_t)HID * 4 + 3 * kMpD * 4 + (size_t)kMpOutWarps * 2048 + 32;
  D2S_REQUIRE(smem <= 227 * 1024, D2S_ERR_ARG, "mlp_residual_ln: needs %zu B of shared memory", smem);
  static SmemOptIn opt, opt_ln;
  cudaError_t e = in_stats ? opt_in_smem(opt_ln, mlp_pair_kernel<true>, 227 * 1024) : opt_in_smem(opt, mlp_pair_kernel<false>, 227 * 1024);
  D2S_REQUIRE(e == cudaSuccess, D2S_ERR_CUDA, "mlp_residual_ln: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  const int pair_tiles = (M + 2 * kMpBM - 1) / (2 * kMpBM);
  const int pairs = pair_tiles < kNumSMs / 2 ? pair_tiles : kNumSMs / 2;
  if (in_stats) mlp_pair_kernel<true><<<2 * pairs, kMpThreads, smem, (cudaStream_t)stream>>>(ma, mw1, mw2, p);
  else          mlp_pair_kernel<false><<<2 * pairs, kMpThreads, smem, (cudaStream_t)stream>>>(ma, mw1, mw2, p);
  count_launch();
  return check_launch(what);
}

extern "C" int d2s_mlp_residual_ln_bf16(const void* h, const void* w1, const void* b1, const void* w2, const void* b2,
                                        const void* x, const void* gamma, const void* beta, float eps, int M, int D, int HID,
                                        int T, int norm_row0, void* out_sum, void* out_norm, d2s_stream_t stream) {
  return mp_launch("d2s_mlp_residual_ln_bf16", h, nullptr, nullptr, nullptr, w1, b1, w2, b2, x, gamma, beta, eps, M, D, HID, T, norm_row0,
                   out_sum, out_norm, nullptr, stream);
}

extern "C" int d2s_mlp_lnin_residual_ln_bf16(const void* x, const float* in_stats, const void* in_gamma, const void* in_beta,
                                             const void* w1, const void* b1, const void* w2, const void* b2, const void* gamma,
                                             const void* beta, float eps, int M, int D, int HID, int T, int norm_row0, void* out_sum,
                                             void* out_norm, float* out_stats, d2s_stream_t stream) {
  D2S_REQUIRE((reinterpret_cast<uintptr_t>(out_stats) & 7u) == 0, D2S_ERR_ALIGN, "mlp_lnin_residual_ln: out_stats must be 8-byte aligned");
  D2S_REQUIRE(in_stats && in_gamma && in_beta && (reinterpret_cast<uintptr_t>(in_stats) & 7u) == 0, D2S_ERR_ARG,
              "mlp_lnin_residual_ln: in_stats (M,2) f32 (8-byte aligned), in_gamma and in_beta are required");
  return mp_launch("d2s_mlp_lnin_residual_ln_bf16", x, in_stats, in_gamma, in_beta, w1, b1, w2, b2, x, gamma, beta, eps, M, D, HID, T,
                   norm_row0, out_sum, out_norm, out_stats, stream);
}
