// CTA-pair (tcgen05 cta_group::2) GEMMs of Block.forward with the neighbouring elementwise work in the epilogue
// (vit_models/dynamic_vit.py:263-283, Mlp.forward :159-175; SURVEY.md section 8f rank 1):
//
//   MODE_LN   x' = x + (A @ W^T + bias);  h = LayerNorm(x') * gamma + beta          (attn.proj / mlp.fc2 + residual + next norm)
//   MODE_ACT  out = act(A @ W^T + bias)                                             (mlp.fc1 + GELU)
//
// bf16 operands, fp32 accumulation in TMEM, every intermediate rounded to bf16 exactly where the reference's separate
// Linear / add / LayerNorm kernels round (Linear output, residual sum), LayerNorm statistics in fp32.
//
// Two CTAs of a cluster (one TPC) work on a 256-row tile: each CTA loads its own 128 rows of A and HALF of the W tile;
// one thread of the leader CTA issues tcgen05.mma.cta_group::2 (M = 256), which reads A and W from both CTAs' shared
// memory and leaves each CTA's 128 x N accumulator in its own TMEM.  Against one-CTA tiles this halves the W traffic
// from L2 per FLOP (the L2 -> SM path, ~42 B/clk/SM, is what bounds a 128-row tile at K = 384) and the shared-memory
// operand reads per MMA.
//
//   warp 0     TMA producer (both CTAs): A 128x64 + W (N/2)x64 bf16 boxes, SWIZZLE_128B, ring of stages; completion is
//              signalled on the LEADER's `full` barrier (cp.async.bulk.tensor ... .cta_group::2)
//   warp 1     TMEM allocation (both CTAs); MMA issue (leader only); tcgen05.commit multicast frees the ring slot in
//              both CTAs and publishes the accumulator to both epilogues
//   warps 2-17 epilogue (both CTAs), four warps per TMEM lane quadrant splitting the columns
//
// MODE_LN keeps the whole 128 x D row tile (D = 192 or 384 <= 512 TMEM columns; D = 768 as two 384-column halves accumulated
// one after the other, the first normalised from its own freshly written x' lines) in the CTA, so the LayerNorm of the
// freshly produced residual stream is computed in the same kernel.  Each epilogue thread owns one row and half of its
// columns and keeps them in registers: the residual rows are fetched with coalesced loads while the MMAs still run and
// transposed to one-row-per-lane through a 4 KB per-warp buffer; pass 1 reads the accumulator, forms x' and the fp32
// sum / sum of squares and releases TMEM (the next tile's MMAs start here); x' goes out through the same per-warp
// transposition as coalesced 128-byte lines; pass 2 normalises the registers and writes h the same way.  (A row far off zero
// gets two-pass statistics from its freshly written x' lines instead of the one-pass sums: see the statistics below.)  No
// CTA-wide barrier and no tile-sized staging buffer: shared memory goes to a 4-deep operand ring instead (a 96 KB
// residual tile left only 3 stages = 48 KB of A in flight per SM, too little to cover HBM latency at K = 1536).
// The separate add+LayerNorm kernel (8 bytes of traffic per element) and the GEMM's own output round trip disappear.
#include <stdlib.h>
#include "d2s_tc.cuh"

namespace d2s {

constexpr int kGpBM = 128, kGpBK = 64, kGpMaxThreads = 576;   // warp 0 TMA, warp 1 MMA, warps 2.. epilogue (4 x PARTS of them)
constexpr uint32_t kGpABytes = kGpBM * 128;      // 128 rows x 64 bf16
constexpr uint32_t kGpBlkBytes = 128 * 128;      // one staged 128 x 64 bf16 block (SWIZZLE_128B)

enum { kGpModeAct = 0, kGpModeLn = 1, kGpModeAct192 = 2 };   // Act192: MODE_ACT with 192-column tiles (N % 192 == 0, e.g. N = 384)

// clock64 phase totals per epilogue warp (profiling builds only: D2S_NVCC_EXTRA=-DD2S_GEMM_TRACE_BUILD; buffer named by D2S_GEMM_TRACE)
#ifdef D2S_GEMM_TRACE_BUILD
#define GP_TRACE_DECL(n) long long tr[n] = {}; long long tr_t = clock64();
#define GP_TRACE(i) { const long long tr_n = clock64(); tr[i] += tr_n - tr_t; tr_t = tr_n; }
#define GP_TRACE_DUMP(n, tiles) if (p.trace && lane == 0) { long long* dst = p.trace + ((size_t)blockIdx.x * 16 + ew) * 8; \
    for (int i = 0; i < n; ++i) dst[i] = tr[i]; dst[7] = tiles; }
#else
#define GP_TRACE_DECL(n)
#define GP_TRACE(i)
#define GP_TRACE_DUMP(n, tiles)
#endif

template <int MODE, int NSUB> struct GpCfg;
template <> struct GpCfg<kGpModeAct, 1> {        // fc1: 256-column tiles, accumulator double-buffered
  static constexpr int UN = 256, NSUB = 1, ACC = 2, STAGES = 4, BLOCKS = 4;      // BLOCKS: staging blocks of 16 KB
  static constexpr int PARTS = 4, MAXREG = 96;     // epilogue warps per TMEM lane quadrant; 2 + 16 warps -> 20 allocated -> 102 regs
};
template <> struct GpCfg<kGpModeAct192, 1> {     // qkv (N = 1152) and the predictors' Linear(D, D) + GELU (N = 384): 192-column tiles,
  static constexpr int UN = 192, NSUB = 1, ACC = 2, STAGES = 6, BLOCKS = 3;      // accumulator double-buffered.  6 x 28 KB of ring =
  static constexpr int PARTS = 3, MAXREG = 128;    // 96 KB of RESIDENT A rows + 6 x 12 KB of W ring when K <= 384 (p.ares)
};
template <> struct GpCfg<kGpModeLn, 2> {         // D = 384: two N = 192 MMAs per k-step, one accumulator
  static constexpr int UN = 192, NSUB = 2, ACC = 1, STAGES = 4, BLOCKS = 3;
  static constexpr int PARTS = 3, MAXREG = 128;    // 2 + 12 warps -> 16 allocated -> 128 regs: a thread keeps 4 chunks (64 regs) of its row
};
template <> struct GpCfg<kGpModeLn, 1> {         // D = 192
  static constexpr int UN = 192, NSUB = 1, ACC = 1, STAGES = 4, BLOCKS = 3;
  static constexpr int PARTS = 3, MAXREG = 128;
};

struct GpBars {
  uint64_t full[6], empty[6], tmem_full[2], tmem_empty[2], a_full[6], a_empty[6], a_ready[6];
  uint32_t tmem_base;
  uint32_t pad;
};

struct GpParams {
  const __nv_bfloat16* bias;    // (N) or NULL
  const __nv_bfloat16* gamma;   // MODE_LN: (N) or NULL when no LayerNorm output is wanted
  const __nv_bfloat16* beta;
  const __nv_bfloat16* x;       // MODE_LN: residual input (M,N)
  __nv_bfloat16* out_sum;       // MODE_LN: x' (M,N)
  __nv_bfloat16* out_norm;      // MODE_LN: LayerNorm(x') (M,N) or NULL
  __nv_bfloat16* pre;           // MODE_ACT: the pre-activation A @ W^T + bias (M,N) as a second output, or NULL
  float2* stats;                // MODE_LN: per-row (mean, rstd) of x' (M), or NULL -- lets the consumer apply the LayerNorm itself
  float eps;
  int M, N, K, act, want_ln;
  long long* trace;             // D2S_GEMM_TRACE: device buffer for per-warp clock64 phase totals (profiling only)
  int ares;                     // MODE_ACT192, K <= 384: the row tile's A rows stay resident across its column tiles
  int groups;                   // MODE_ACT*: a row tile's column tiles are split into `groups` work units (last-wave quantisation); 1 otherwise
  // MODE_ACT192 + ares: LayerNorm of the INPUT rows applied on the fly (A is the raw residual stream, in_stats its per-row (mean, rstd))
  const float2* in_stats;
  const __nv_bfloat16 *in_gamma, *in_beta;
};

// Sum of (x - m)^2 over `nblk` 64-column blocks of one bf16 row, `stride` elements apart (the rare two-pass statistics of a
// row far off zero; out of line, so that the epilogue keeps its registers)
__device__ __noinline__ float bf16_sq_dev_blocks(const __nv_bfloat16* x, int nblk, int stride, float m) {
  const uint64_t nm = f2_bcast(-m);
  uint64_t acc0 = f2_bcast(0.f), acc1 = f2_bcast(0.f);
  for (int b = 0; b < nblk; ++b)
#pragma unroll 2
    for (int k = 0; k < 8; ++k) {
      const uint4 t = ld_cg16(x + (size_t)b * stride + k * 8);
      const uint64_t d0 = f2_add(f2_pack(bf16_lo(t.x), bf16_hi(t.x)), nm), d1 = f2_add(f2_pack(bf16_lo(t.y), bf16_hi(t.y)), nm);
      const uint64_t d2 = f2_add(f2_pack(bf16_lo(t.z), bf16_hi(t.z)), nm), d3 = f2_add(f2_pack(bf16_lo(t.w), bf16_hi(t.w)), nm);
      acc0 = f2_fma(d2, d2, f2_fma(d0, d0, acc0));
      acc1 = f2_fma(d3, d3, f2_fma(d1, d1, acc1));
    }
  float a0, a1, b0, b1;
  f2_unpack(acc0, a0, a1);
  f2_unpack(acc1, b0, b1);
  return (a0 + a1) + (b0 + b1);
}

template <int MODE, int NSUB_, int ACT>
__global__ void __cluster_dims__(2, 1, 1) __maxnreg__((GpCfg<MODE, NSUB_>::MAXREG))
gemm_pair_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
                 const __grid_constant__ CUtensorMap map_o,    // MODE_ACT: output (TMA store)
                 const GpParams p) {
  using Cfg = GpCfg<MODE, NSUB_>;
  constexpr int UN = Cfg::UN, NSUB = Cfg::NSUB, ACC = Cfg::ACC, STAGES = Cfg::STAGES, PARTS = Cfg::PARTS;
  constexpr int kThreads = (2 + 4 * PARTS) * 32;
  constexpr int TN = UN * NSUB;                                 // output columns per tile
  constexpr uint32_t kBSub = (UN / 2) * 128;                    // this CTA's half of one W sub-tile
  constexpr uint32_t kStage = kGpABytes + NSUB * kBSub;
  constexpr uint32_t kAccCols = (TN <= 256) ? 256 : 512;        // TMEM columns per accumulator stage

  extern __shared__ unsigned char smem_dyn[];
  const uint32_t raw = smem_u32(smem_dyn);
  const uint32_t padb = (1024u - (raw & 1023u)) & 1023u;
  unsigned char* ring = smem_dyn + padb;
  unsigned char* blocks = ring + STAGES * kStage;               // MODE_ACT: store staging; MODE_LN: x / x' / h tile
  GpBars* bars = reinterpret_cast<GpBars*>(blocks + Cfg::BLOCKS * kGpBlkBytes);
  float* bias_s = reinterpret_cast<float*>(bars + 1);           // N floats (MODE_ACT) / 3 x N floats (MODE_LN)
  float2* red_s = reinterpret_cast<float2*>(bias_s + (MODE == kGpModeLn ? 3 * p.N : p.N));   // MODE_LN: [PARTS][128] partial stats
  volatile uint32_t* sel_s = reinterpret_cast<volatile uint32_t*>(red_s + 4 * 128);           // MODE_LN: byte-permute selectors
  uint32_t* gbin_s = reinterpret_cast<uint32_t*>(bias_s + p.N);                               // MODE_ACT192, in_stats: K x (gamma, beta) as bf16 pairs

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int pair_tiles = (p.M + 2 * kGpBM - 1) / (2 * kGpBM);
  const int n_tiles = p.N / TN, k_blocks = p.K / kGpBK;
  const int G = MODE == kGpModeLn ? 1 : p.groups, npg = n_tiles / G, units = pair_tiles * G;   // work unit = (row tile, group of npg column tiles)

  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(smem_u32(&bars->full[i]), 1); mbar_init(smem_u32(&bars->empty[i]), 1); }
    for (int i = 0; i < 6; ++i) {
      mbar_init(smem_u32(&bars->a_full[i]), 1);
      mbar_init(smem_u32(&bars->a_empty[i]), 1);
      mbar_init(smem_u32(&bars->a_ready[i]), 2 * 4 * PARTS);      // in_stats: every epilogue warp of both CTAs has normalised its share
    }
    for (int i = 0; i < 2; ++i) { mbar_init(smem_u32(&bars->tmem_full[i]), 1); mbar_init(smem_u32(&bars->tmem_empty[i]), 8 * PARTS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (MODE == kGpModeLn) { sel_s[0] = 0x1044u; sel_s[1] = 0x3244u; }   // {0, 0, b0, b1} and {0, 0, b2, b3}
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  if (MODE == kGpModeLn) {
    for (int i = tid; i < p.N; i += kThreads) {
      bias_s[i] = p.bias ? __bfloat162float(p.bias[i]) : 0.f;
      bias_s[p.N + i] = p.gamma ? __bfloat162float(p.gamma[i]) : 1.f;
      bias_s[2 * p.N + i] = p.beta ? __bfloat162float(p.beta[i]) : 0.f;
    }
  } else {
    for (int i = tid; i < p.N; i += kThreads) bias_s[i] = p.bias ? __bfloat162float(p.bias[i]) : 0.f;
    if (MODE == kGpModeAct192 && p.in_stats)
      for (int i = tid; i < p.K; i += kThreads)
        gbin_s[i] = (uint32_t)__bfloat16_as_ushort(p.in_gamma[i]) | ((uint32_t)__bfloat16_as_ushort(p.in_beta[i]) << 16);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;

  if (warp == 0) {
    if (lane == 0) {
      // ======================================= TMA producer (both CTAs) =======================================
      uint32_t it = 0;
      if (MODE == kGpModeAct192 && p.ares) {
        // A resident: the row tile's k-blocks are loaded ONCE (each as soon as the previous tile's last column tile has read
        // it) and every column tile streams only its W blocks: per row tile 96 + n_tiles x 72 KB through the SM's L2 port
        // instead of n_tiles x 168 KB
        unsigned char* wring = ring + 6 * kGpABytes;
        uint32_t at = 0;
        for (int un = pair; un < units; un += num_pairs, ++at) {
          const int pt = un / G, nt0 = (un - pt * G) * npg;
          const int row0 = pt * 2 * kGpBM + (int)rank * kGpBM;
          for (int kb = 0; kb < k_blocks; ++kb) {
            mbar_wait(smem_u32(&bars->a_empty[kb]), (at & 1) ^ 1);
            const uint32_t af = smem_u32(&bars->a_full[kb]);
            if (p.in_stats) {     // each CTA's own barrier: its epilogue warps normalise the block before the pair's MMAs read it
              mbar_expect_tx(af, kGpABytes);
              tma_load_2d(smem_u32(ring + kb * kGpABytes), &map_a, kb * kGpBK, row0, af);
            } else {
              if (rank == 0) mbar_expect_tx(af, 2 * kGpABytes);
              tma_load_2d_pair(smem_u32(ring + kb * kGpABytes), &map_a, kb * kGpBK, row0, mapa(af, 0));
            }
          }
          for (int nt = nt0; nt < nt0 + npg; ++nt)
            for (int kb = 0; kb < k_blocks; ++kb, ++it) {
              const uint32_t s = it % STAGES, n = it / STAGES;
              mbar_wait(smem_u32(&bars->empty[s]), (n & 1) ^ 1);
              const uint32_t full_local = smem_u32(&bars->full[s]);
              if (rank == 0) mbar_expect_tx(full_local, 2 * kBSub);
              tma_load_2d_pair(smem_u32(wring + s * kBSub), &map_w, kb * kGpBK, nt * TN + (int)rank * (UN / 2), mapa(full_local, 0));
            }
        }
      } else
      for (int un = pair; un < units; un += num_pairs) {
        const int pt = un / G, nt0 = (un - pt * G) * npg;
        const int row0 = pt * 2 * kGpBM + (int)rank * kGpBM;
        for (int nt = nt0; nt < nt0 + npg; ++nt)
          for (int kb = 0; kb < k_blocks; ++kb, ++it) {
            const uint32_t s = it % STAGES, n = it / STAGES;
            mbar_wait(smem_u32(&bars->empty[s]), (n & 1) ^ 1);
            const uint32_t full_local = smem_u32(&bars->full[s]);
            if (rank == 0) mbar_expect_tx(full_local, 2 * kStage);       // both CTAs' boxes land on the leader's barrier
            const uint32_t full_leader = mapa(full_local, 0);
            const uint32_t dst = smem_u32(ring + s * kStage);
            tma_load_2d_pair(dst, &map_a, kb * kGpBK, row0, full_leader);
#pragma unroll
            for (int j = 0; j < NSUB; ++j)
              tma_load_2d_pair(dst + kGpABytes + j * kBSub, &map_w, kb * kGpBK, nt * TN + j * UN + (int)rank * (UN / 2), full_leader);
          }
      }
    }
  } else if (warp_uniform(warp) == 1) {
    if (warp_uniform((int)rank) == 0) {
      // ===== MMA issuer (leader): the whole warp runs the loop warp-uniformly, one elected lane issues (see elect_one) =====
      const uint32_t idesc = make_idesc(2 * kGpBM, UN, 0);
      uint32_t it = 0, tile = 0;
      for (int un = pair; un < units; un += num_pairs)
        for (int nt = 0; nt < npg; ++nt, ++tile) {                       // (the issuer only needs the position inside the unit)
          const uint32_t as = tile % ACC, an = tile / ACC;
          mbar_wait(smem_u32(&bars->tmem_empty[as]), (an & 1) ^ 1);      // both epilogues have drained this accumulator
          tc_fence_after();
          const uint32_t d = tmem + as * kAccCols;
          const bool ares = MODE == kGpModeAct192 && p.ares;
          const uint32_t at = tile / (uint32_t)npg;                // work units done by this pair
          for (int kb = 0; kb < k_blocks; ++kb, ++it) {
            const uint32_t s = it % STAGES, n = it / STAGES;
            if (ares && nt == 0) mbar_wait(smem_u32(p.in_stats ? &bars->a_ready[kb] : &bars->a_full[kb]), at & 1);
            mbar_wait(smem_u32(&bars->full[s]), n & 1);
            tc_fence_after();
            const uint64_t ad = make_desc_sw128(smem_u32(ares ? ring + kb * kGpABytes : ring + s * kStage), 16, 1024);
            if (elect_one()) {
#pragma unroll
              for (int j = 0; j < NSUB; ++j) {
                const uint64_t bd = make_desc_sw128(smem_u32(ares ? ring + 6 * kGpABytes + s * kBSub : ring + s * kStage + kGpABytes + j * kBSub), 16, 1024);
                if (kb == 0) mma2_ss_imm<false>(d + j * UN, ad, bd, idesc); else mma2_ss_imm<true>(d + j * UN, ad, bd, idesc);
                mma2_ss_imm<true>(d + j * UN, ad + 2, bd + 2, idesc);
                mma2_ss_imm<true>(d + j * UN, ad + 4, bd + 4, idesc);
                mma2_ss_imm<true>(d + j * UN, ad + 6, bd + 6, idesc);
              }
              mma2_commit_both(smem_u32(&bars->empty[s]));               // ring slot free in both CTAs once these retire
              if (ares && nt == npg - 1) mma2_commit_both(smem_u32(&bars->a_empty[kb]));   // the unit's last reader of this A block
            }
            __syncwarp();
          }
          if (elect_one()) mma2_commit_both(smem_u32(&bars->tmem_full[as]));
          __syncwarp();
        }
    }
  } else {
    // ========================================= epilogue (both CTAs) =========================================
    // 4 x PARTS warps: PARTS per TMEM lane quadrant (a warp may only touch lanes 32 (warp % 4) ...), each taking 1/PARTS of the columns
    const int ew = warp - 2;                    // 0..4*PARTS-1
    const int quad = warp & 3;                  // TMEM lane quadrant of this warp
    const int part = ew >> 2;                   // which share of the columns
    const int r = quad * 32 + lane;             // row inside this CTA's 128-row tile
    const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16);
    uint32_t tile = 0;

    if (MODE != kGpModeLn) {
      // part p owns the 64-column block p of every 256- (192-) column tile: one staging block, one TMA store per tile
      GP_TRACE_DECL(5)
      const bool issuer = (ew & 3) == 0 && lane == 0;
      unsigned char* blk = blocks + (size_t)part * kGpBlkBytes;
      // in_stats (A resident): the unit's input rows arrive as the raw residual stream; this thread normalises its row's share of
      // every k-block in place, h = bf16(((x - mean) * rstd) * gamma + beta) -- the arithmetic of the LayerNorm pass of MODE_LN, so
      // the operand is bit-identical to the normalised copy the producer no longer writes.  The NEXT unit's blocks are handled in
      // front of the current unit's last column tile (they land as soon as that tile's MMAs have retired); the kernel is bound
      // by its stores, so the MMA pipe's short wait for a_ready is hidden.
      const bool lnin = MODE == kGpModeAct192 && p.ares && p.in_stats != nullptr;
      auto normalize_unit = [&](int un_n, uint32_t at_n) {
        const int row = (un_n / G) * 2 * kGpBM + (int)rank * kGpBM + r;
        const float2 st = row < p.M ? p.in_stats[row] : make_float2(0.f, 0.f);
        const uint64_t sc = f2_bcast(st.y), sh = f2_bcast(-st.x * st.y);
#pragma unroll 1
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(smem_u32(&bars->a_full[kb]), at_n & 1);
          unsigned char* hb = ring + kb * kGpABytes;
          for (int ch = part; ch < 8; ch += PARTS) {
            uint4* ptr = reinterpret_cast<uint4*>(hb + sw128_off(r, ch));
            const uint4 t = *ptr;
            const uint32_t w[4] = {t.x, t.y, t.z, t.w};
            uint32_t o[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const uint2 gb = *reinterpret_cast<const uint2*>(&gbin_s[kb * 64 + ch * 8 + 2 * q]);
              float h0, h1;
              f2_unpack(f2_fma(f2_fma(f2_pack(bf16_lo(w[q]), bf16_hi(w[q])), sc, sh), f2_pack(bf16_lo(gb.x), bf16_lo(gb.y)),
                               f2_pack(bf16_hi(gb.x), bf16_hi(gb.y))), h0, h1);
              o[q] = pack_bf16x2(h0, h1);
            }
            *ptr = make_uint4(o[0], o[1], o[2], o[3]);
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(mapa(smem_u32(&bars->a_ready[kb]), 0));
        }
      };
      uint32_t at = 0;
      if (lnin && pair < units) normalize_unit(pair, 0);
      for (int un = pair; un < units; un += num_pairs, ++at) {
        const int pt = un / G, nt0 = (un - pt * G) * npg;
        const int row0 = pt * 2 * kGpBM + (int)rank * kGpBM;
        for (int nt = nt0; nt < nt0 + npg; ++nt, ++tile) {
          if (lnin && nt == nt0 + npg - 1 && un + num_pairs < units) normalize_unit(un + num_pairs, at + 1);
          const uint32_t as = tile % ACC, an = tile / ACC;
          mbar_wait(smem_u32(&bars->tmem_full[as]), an & 1);
          tc_fence_after();
          GP_TRACE(0)
          const int col0 = nt * TN + part * 64;
          const uint32_t taddr = lane_addr + as * kAccCols + part * 64;
          // the TMA store that last read this block (previous tile) must be done before it is overwritten
          if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          asm volatile("bar.sync %0, 128;" ::"r"(1 + part) : "memory");
          GP_TRACE(1)
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            uint32_t v[32];
            tmem_ld32_nowait(taddr + c * 32, v);
            tmem_ld_wait();
            GP_TRACE(2)
            uint32_t o[16];
            // training: the Linear's own output is a second result (GELU' needs it); one 64-byte row segment per thread,
            // straight from registers (no room for a second staging block next to a 4-stage operand ring)
            const bool want_pre = p.pre != nullptr;
            const bool row_ok = row0 + r < p.M;
            __nv_bfloat16* pre_row = p.pre + (size_t)(row_ok ? row0 + r : 0) * p.N + col0 + c * 32;
            uint32_t pw[8];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              const float2 bq = *reinterpret_cast<const float2*>(&bias_s[col0 + c * 32 + 2 * q]);
              uint64_t xp = f2_add(f2_pack(__uint_as_float(v[2 * q]), __uint_as_float(v[2 * q + 1])), f2_pack(bq.x, bq.y));
              float x0, x1;
              if (want_pre) {
                f2_unpack(xp, x0, x1);
                pw[q & 7] = pack_bf16x2(x0, x1);
                if ((q & 7) == 7 && row_ok) st_global_v8(pre_row + (q >> 3) * 16, pw);     // whole 32-byte sectors
              }
              if (ACT == D2S_ACT_GELU) xp = gelu_erf_pair(xp);
              f2_unpack(xp, x0, x1);
              if (ACT == D2S_ACT_RELU) { x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); }
              o[q] = pack_bf16x2(x0, x1);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q)
              *reinterpret_cast<uint4*>(blk + sw128_off(r, c * 4 + q)) = make_uint4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
            GP_TRACE(3)
          }
          // all TMEM reads of this accumulator are done: hand it back before the store drains
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(mapa(smem_u32(&bars->tmem_empty[as]), 0));
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          asm volatile("bar.sync %0, 128;" ::"r"(1 + part) : "memory");
          if (issuer) {
            tma_store_2d(&map_o, smem_u32(blk), col0, row0);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
          GP_TRACE(4)
        }
      }
      GP_TRACE_DUMP(5, tile)
    } else {
      // ---- MODE_LN: rows of N = n_tiles x TN columns (n_tiles = 1: D = 192 / 384; n_tiles = 2: D = 768, whose 128 x 768 fp32
      // row tile does not fit the 512 TMEM columns: the two 384-column halves are accumulated one after the other).  This
      // thread owns row r and the 64-column blocks b = PARTS bi + part of the current half (whole 128-byte lines), and keeps
      // its x / x' values in registers (BPT x 32 packed bf16 pairs); the row statistics run on across the halves.  After the
      // last half the registers hold that half's x'; earlier halves are normalised from the x' lines this warp itself wrote
      // a moment ago (L2 hits), in the coalesced layout, with mean / rstd fetched from the owning lane by shuffle. ----
      constexpr int NBLK = TN / 64, BPT = NBLK / PARTS;
      static_assert(MODE != kGpModeLn || NBLK % PARTS == 0, "column blocks must split evenly over the epilogue warps");
      const int ldn = p.N;
      const float* gamma_s = bias_s + ldn;
      const float* beta_s = bias_s + 2 * ldn;
      unsigned char* buf = blocks + ew * 4096;                  // per-warp [32 rows x 128 B] transposition buffer
      const int crow = lane >> 3, cseg = lane & 7;              // coalesced pattern: 8 lanes x 16 B cover one row's 128-byte line
      const uint32_t co_off = (uint32_t)crow * 128, co_seg = (uint32_t)cseg;
      const uint32_t own_off = (uint32_t)lane * 128, own_sw = (uint32_t)lane & 7u;
      GP_TRACE_DECL(7)
      for (int pt = pair; pt < pair_tiles; pt += num_pairs) {
        const int row0 = pt * 2 * kGpBM + (int)rank * kGpBM + quad * 32;     // first row of this warp
        uint32_t xr[BPT][32];      // this thread's values, 2 bf16 per word: first in the coalesced layout, then its own row
        // element offset of (row0 + crow, column part*64 + cseg*8); half nt / block bi / row group i add on top
        const size_t goff = (size_t)(row0 + crow) * ldn + part * 64 + cseg * 8;
        const int rows_left = p.M - row0 - crow;                  // row group i is in range iff 4 i < rows_left
        uint64_t acc_s = f2_bcast(0.f), acc_q = f2_bcast(0.f);
        for (int nt = 0; nt < n_tiles; ++nt, ++tile) {
          const int cb = nt * TN;                                 // first column of this half
          // ---- residual rows: coalesced loads (issued before the accumulator is awaited), transposed to one row per lane ----
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            // rows past M re-read the last valid row (their results are never stored): no predicated loads, no zero fills
            const int grow = min(row0 + crow + 4 * i, p.M - 1);
            const __nv_bfloat16* xp = p.x + (size_t)grow * ldn + cb + part * 64 + cseg * 8;
#pragma unroll
            for (int bi = 0; bi < BPT; ++bi) {
              const uint4 t = ld_nc16(xp + bi * (PARTS * 64));
              xr[bi][4 * i] = t.x; xr[bi][4 * i + 1] = t.y; xr[bi][4 * i + 2] = t.z; xr[bi][4 * i + 3] = t.w;
            }
          }
#pragma unroll
          for (int bi = 0; bi < BPT; ++bi) {
#pragma unroll
            for (int i = 0; i < 8; ++i)    // row 4 i + crow: (row & 7) = ((4 i) & 7) + crow
              *reinterpret_cast<uint4*>(buf + co_off + i * 512 + ((co_seg ^ (uint32_t)((4 * i + crow) & 7)) << 4)) =
                  make_uint4(xr[bi][4 * i], xr[bi][4 * i + 1], xr[bi][4 * i + 2], xr[bi][4 * i + 3]);
            __syncwarp();
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const uint4 t = *reinterpret_cast<const uint4*>(buf + own_off + (((uint32_t)q ^ own_sw) << 4));
              xr[bi][4 * q] = t.x; xr[bi][4 * q + 1] = t.y; xr[bi][4 * q + 2] = t.z; xr[bi][4 * q + 3] = t.w;
            }
            __syncwarp();
          }
          GP_TRACE(0)
          mbar_wait(smem_u32(&bars->tmem_full[0]), tile & 1);
          tc_fence_after();
          GP_TRACE(1)
          // ---- pass 1: x' = bf16(x + bf16(acc + bias)) in registers, fp32 sum / sum of squares of the rounded values ----
#pragma unroll
          for (int bi = 0; bi < BPT; ++bi) {
            const int col0 = (PARTS * bi + part) * 64;
#pragma unroll
            for (int hh = 0; hh < 4; ++hh) {
              uint32_t v[16];
              tmem_ld16_nowait(lane_addr + col0 + hh * 16, v);
              tmem_ld_wait();
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const float2 bq = *reinterpret_cast<const float2*>(&bias_s[cb + col0 + hh * 16 + 2 * q]);
                float y0, y1;
                f2_unpack(f2_add(f2_pack(__uint_as_float(v[2 * q]), __uint_as_float(v[2 * q + 1])), f2_pack(bq.x, bq.y)), y0, y1);
                const uint32_t yb = pack_bf16x2(y0, y1);                  // the Linear's bf16 output
                // the residual add's bf16 output, x + y rounded once (add.rn.bf16x2).  Working on the packed words also keeps
                // ptxas from unpacking the whole row to fp32 ahead of the accumulator wait (2x the live registers -> spills).
                const uint32_t sb = add_bf16x2(xr[bi][hh * 8 + q], yb);
                xr[bi][hh * 8 + q] = sb;
                const uint64_t sv = f2_pack(bf16_lo(sb), bf16_hi(sb));
                acc_s = f2_add(acc_s, sv);
                acc_q = f2_fma(sv, sv, acc_q);
              }
            }
          }
          // accumulator drained: the next half's / tile's MMAs may start
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(mapa(smem_u32(&bars->tmem_empty[0]), 0));
          GP_TRACE(2)
          // ---- x' out: one row per lane -> coalesced 128-byte lines ----
#pragma unroll
          for (int bi = 0; bi < BPT; ++bi) {
#pragma unroll
            for (int q = 0; q < 8; ++q)
              *reinterpret_cast<uint4*>(buf + own_off + (((uint32_t)q ^ own_sw) << 4)) =
                  make_uint4(xr[bi][4 * q], xr[bi][4 * q + 1], xr[bi][4 * q + 2], xr[bi][4 * q + 3]);
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const uint4 val = *reinterpret_cast<const uint4*>(buf + co_off + i * 512 + ((co_seg ^ (uint32_t)((4 * i + crow) & 7)) << 4));
              if (4 * i < rows_left) *reinterpret_cast<uint4*>(p.out_sum + goff + (size_t)4 * i * ldn + cb + bi * (PARTS * 64)) = val;
            }
            __syncwarp();
          }
          GP_TRACE(3)
        }
        if (p.want_ln) {
          {
            float s0, s1, q0, q1;
            f2_unpack(acc_s, s0, s1);
            f2_unpack(acc_q, q0, q1);
            red_s[part * 128 + r] = make_float2(s0 + s1, q0 + q1);
          }
          asm volatile("bar.sync %0, %1;" ::"r"(1 + quad), "n"(32 * PARTS) : "memory");     // the warps of this lane quadrant
          float sum = 0.f, sq = 0.f;
#pragma unroll
          for (int k = 0; k < PARTS; ++k) { const float2 t = red_s[k * 128 + r]; sum += t.x; sq += t.y; }
          const float inv_n = 1.0f / (float)ldn;
          float mean = sum * inv_n;
          const float var = fmaxf(sq * inv_n - mean * mean, 0.f);
          float rstd = rsqrtf(var + p.eps);
          const uint32_t sel_lo = sel_s[0], sel_hi = sel_s[1];
          asm volatile("bar.sync %0, %1;" ::"r"(1 + quad), "n"(32 * PARTS) : "memory");     // red_s may be rewritten
          // E[x^2] - mean^2 is exact enough while 8 mean^2 <= var (the sum of squares is then at most 1.125 x the squared
          // deviations).  A row farther off zero would lose log2(1 + mean^2 / var) bits to the cancellation: it gets two-pass
          // statistics instead, from the x' this warp has just written (every lane re-reads its own row, its part's columns).
          // The warps of a lane quadrant hold the same rows and the same sums, so they all take this branch or none.
          const bool far = row0 + lane < p.M && 8.f * mean * mean > var;
          if (far) mean = fmaf(fmaf(-mean, (float)ldn, sum), inv_n, mean);     // sum / N: exact when representable (constant rows)
          if (__any_sync(0xffffffffu, far)) {
            red_s[part * 128 + r].x = far ? bf16_sq_dev_blocks(p.out_sum + (size_t)(row0 + lane) * ldn + part * 64, n_tiles * BPT,
                                                               PARTS * 64, mean) : 0.f;
            asm volatile("bar.sync %0, %1;" ::"r"(1 + quad), "n"(32 * PARTS) : "memory");
            float m2 = 0.f;
#pragma unroll
            for (int k = 0; k < PARTS; ++k) m2 += red_s[k * 128 + r].x;
            asm volatile("bar.sync %0, %1;" ::"r"(1 + quad), "n"(32 * PARTS) : "memory");
            if (far) rstd = rsqrtf(m2 * inv_n + p.eps);
          }
          const uint64_t sc = f2_bcast(rstd), sh = f2_bcast(-mean * rstd);
          if (p.stats != nullptr && part == 0 && row0 + lane < p.M) p.stats[row0 + lane] = make_float2(mean, rstd);
          GP_TRACE(4)
          if (p.out_norm != nullptr) {
          // ---- pass 2: h = (x' - mean) * rstd * gamma + beta for the half in registers (the last one), then out like x' ----
          const int cb_last = (n_tiles - 1) * TN;
#pragma unroll
          for (int bi = 0; bi < BPT; ++bi) {
            const int col0 = cb_last + (PARTS * bi + part) * 64;
#pragma unroll
            for (int q = 0; q < 32; ++q) {
              const float2 g = *reinterpret_cast<const float2*>(&gamma_s[col0 + 2 * q]);
              const float2 bt = *reinterpret_cast<const float2*>(&beta_s[col0 + 2 * q]);
              float h0, h1;
              const uint32_t xv = xr[bi][q];
              // bf16 -> fp32 by byte permutes whose selectors were loaded after the barrier: a true dependency, so the
              // unpack of the whole row cannot be scheduled ahead of its use (again: 2x the live registers)
              const uint64_t xf = f2_pack(__uint_as_float(__byte_perm(xv, 0, sel_lo)), __uint_as_float(__byte_perm(xv, 0, sel_hi)));
              f2_unpack(f2_fma(f2_fma(xf, sc, sh), f2_pack(g.x, g.y), f2_pack(bt.x, bt.y)), h0, h1);
              xr[bi][q] = pack_bf16x2(h0, h1);
            }
#pragma unroll
            for (int q = 0; q < 8; ++q)
              *reinterpret_cast<uint4*>(buf + own_off + (((uint32_t)q ^ own_sw) << 4)) =
                  make_uint4(xr[bi][4 * q], xr[bi][4 * q + 1], xr[bi][4 * q + 2], xr[bi][4 * q + 3]);
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const uint4 val = *reinterpret_cast<const uint4*>(buf + co_off + i * 512 + ((co_seg ^ (uint32_t)((4 * i + crow) & 7)) << 4));
              if (4 * i < rows_left) *reinterpret_cast<uint4*>(p.out_norm + goff + (size_t)4 * i * ldn + cb_last + bi * (PARTS * 64)) = val;
            }
            __syncwarp();
          }
          // ---- earlier halves: x' back from the lines this warp stored above (each lane re-reads exactly the 16-byte pieces
          // it wrote itself), normalised in the coalesced layout ----
          for (int nt = 0; nt + 1 < n_tiles; ++nt) {
            const int cb = nt * TN;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float m_i = __shfl_sync(0xffffffffu, mean, 4 * i + crow), r_i = __shfl_sync(0xffffffffu, rstd, 4 * i + crow);
              const float sh_i = -m_i * r_i;
              if (4 * i < rows_left) {
#pragma unroll
                for (int bi = 0; bi < BPT; ++bi) {
                  const size_t off = goff + (size_t)4 * i * ldn + cb + bi * (PARTS * 64);
                  const uint4 t = *reinterpret_cast<const uint4*>(p.out_sum + off);
                  const int col = cb + (PARTS * bi + part) * 64 + cseg * 8;
                  const uint32_t w[4] = {t.x, t.y, t.z, t.w};
                  uint32_t o[4];
#pragma unroll
                  for (int q = 0; q < 4; ++q) {
                    const float2 g = *reinterpret_cast<const float2*>(&gamma_s[col + 2 * q]);
                    const float2 bt = *reinterpret_cast<const float2*>(&beta_s[col + 2 * q]);
                    // the form of the last half (and of every bf16 LayerNorm producer): fma(fma(x, rstd, -mean rstd), gamma, beta)
                    o[q] = pack_bf16x2(fmaf(fmaf(bf16_lo(w[q]), r_i, sh_i), g.x, bt.x), fmaf(fmaf(bf16_hi(w[q]), r_i, sh_i), g.y, bt.y));
                  }
                  *reinterpret_cast<uint4*>(p.out_norm + off) = make_uint4(o[0], o[1], o[2], o[3]);
                }
              }
            }
          }
          }
          GP_TRACE(5)
        }
      }
      GP_TRACE_DUMP(7, tile)
    }
  }
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // outstanding TMA stores read shared memory
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();            // the peer may still signal barriers / read operands in this CTA's shared memory
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512) : "memory");
  }
}

static long long* gp_trace() {
  const char* e = getenv("D2S_GEMM_TRACE");
  return e ? reinterpret_cast<long long*>(strtoull(e, nullptr, 10)) : nullptr;
}

static int gp_map_2d(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint32_t box_inner, uint32_t box_outer,
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

template <int MODE, int NSUB, int ACT>
static int gp_launch(const CUtensorMap& ma, const CUtensorMap& mw, const CUtensorMap& mo,
                     const GpParams& p, cudaStream_t stream, const char* what) {
  using Cfg = GpCfg<MODE, NSUB>;
  constexpr uint32_t kStage = kGpABytes + NSUB * (Cfg::UN / 2) * 128;
  const size_t smem = 1024 + (size_t)Cfg::STAGES * kStage + (size_t)Cfg::BLOCKS * kGpBlkBytes + sizeof(GpBars) +
                      (MODE == kGpModeLn ? (size_t)3 * p.N * 4 + 4 * 128 * sizeof(float2) + 16
                                          : (size_t)p.N * 4 + (p.in_stats ? (size_t)p.K * 4 : 0));   // gbin_s: in_stats only
  D2S_REQUIRE(smem <= 227 * 1024, D2S_ERR_ARG, "%s: needs %zu B of shared memory", what, smem);
  static SmemOptIn opt;
  cudaError_t e = opt_in_smem(opt, gemm_pair_kernel<MODE, NSUB, ACT>, 227 * 1024);
  D2S_REQUIRE(e == cudaSuccess, D2S_ERR_CUDA, "%s: cudaFuncSetAttribute: %s", what, cudaGetErrorString(e));
  const int pair_tiles = (p.M + 2 * kGpBM - 1) / (2 * kGpBM);
  const int units = pair_tiles * (MODE == kGpModeLn ? 1 : p.groups);
  const int pairs = units < kNumSMs / 2 ? units : kNumSMs / 2;
  gemm_pair_kernel<MODE, NSUB, ACT><<<2 * pairs, (2 + 4 * Cfg::PARTS) * 32, smem, stream>>>(ma, mw, mo, p);
  count_launch();
  return check_launch(what);
}

}  // namespace d2s

using namespace d2s;

static int gp_linear_act(const char* what, const void* a, const float* in_stats, const void* in_gamma, const void* in_beta,
                         const void* w, const void* bias, int M, int N, int K, int act, void* out, void* pre, d2s_stream_t stream) {
  D2S_REQUIRE(a && w && out, D2S_ERR_ARG, "linear_act_pair: null pointer");
  const bool t192 = N % 256 != 0;                  // 192-column tiles for widths like 384
  D2S_REQUIRE(M >= 0 && N >= 192 && (N % 256 == 0 || N % 192 == 0) && N <= 4096 && K >= kGpBK && K % kGpBK == 0, D2S_ERR_ARG,
              "linear_act_pair: need N %% 256 == 0 or N %% 192 == 0 (N <= 4096) and K %% %d == 0 (got M=%d N=%d K=%d)", kGpBK, M, N, K);
  D2S_REQUIRE(act >= D2S_ACT_NONE && act <= D2S_ACT_RELU, D2S_ERR_ARG, "linear_act_pair: bad activation %d", act);
  D2S_REQUIRE(aligned16(a) && aligned16(w) && aligned16(out) && aligned16(pre), D2S_ERR_ALIGN,
              "linear_act_pair: pointers must be 16-byte aligned");
  if (M == 0) return D2S_OK;
  CUtensorMap ma, mw, mo;
  int rc;
  if ((rc = gp_map_2d(&ma, a, K, M, kGpBK, kGpBM, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, what))) return rc;
  if ((rc = gp_map_2d(&mw, w, K, N, kGpBK, t192 ? 96 : 128, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, what))) return rc;
  if ((rc = gp_map_2d(&mo, out, N, M, 64, kGpBM, CU_TENSOR_MAP_L2_PROMOTION_NONE, what))) return rc;
  // Split a row tile's column tiles into G work units when that shortens the last wave: time per CTA pair ~
  // ceil(row tiles * G / pairs) units of (column tiles per unit + 0.25) -- each unit (re)loads the A rows, partly exposed.
  const int n_tiles = N / (t192 ? 192 : 256), pair_tiles = (M + 2 * kGpBM - 1) / (2 * kGpBM), np = kNumSMs / 2;
  int groups = 1;
  double best = (double)((pair_tiles + np - 1) / np) * (n_tiles + 0.25);
  for (int g = 2; g <= n_tiles; ++g) {
    if (n_tiles % g) continue;
    const double r = (double)((pair_tiles * g + np - 1) / np) * (n_tiles / g + 0.25);
    if (r < best * 0.99) { best = r; groups = g; }
  }
  GpParams p{(const __nv_bfloat16*)bias, nullptr, nullptr, nullptr, nullptr, nullptr, (__nv_bfloat16*)pre, nullptr, 0.f, M, N, K, act, 0,
             gp_trace(), (t192 && K <= 6 * kGpBK) ? 1 : 0, groups,
             reinterpret_cast<const float2*>(in_stats), (const __nv_bfloat16*)in_gamma, (const __nv_bfloat16*)in_beta};
  D2S_REQUIRE(!in_stats || p.ares, D2S_ERR_ARG, "%s: the on-the-fly input LayerNorm needs N %% 192 == 0 (N %% 256 != 0) and K <= %d", what,
              6 * kGpBK);
  if (t192) {
    if (act == D2S_ACT_GELU) return gp_launch<kGpModeAct192, 1, D2S_ACT_GELU>(ma, mw, mo, p, (cudaStream_t)stream, what);
    if (act == D2S_ACT_RELU) return gp_launch<kGpModeAct192, 1, D2S_ACT_RELU>(ma, mw, mo, p, (cudaStream_t)stream, what);
    return gp_launch<kGpModeAct192, 1, D2S_ACT_NONE>(ma, mw, mo, p, (cudaStream_t)stream, what);
  }
  if (act == D2S_ACT_GELU) return gp_launch<kGpModeAct, 1, D2S_ACT_GELU>(ma, mw, mo, p, (cudaStream_t)stream, what);
  if (act == D2S_ACT_RELU) return gp_launch<kGpModeAct, 1, D2S_ACT_RELU>(ma, mw, mo, p, (cudaStream_t)stream, what);
  return gp_launch<kGpModeAct, 1, D2S_ACT_NONE>(ma, mw, mo, p, (cudaStream_t)stream, what);
}

static int gp_linear_residual(const char* what, const void* a, const void* w, const void* bias, const void* x, const void* gamma,
                              const void* beta, float eps, int M, int N, int K, void* out_sum, void* out_norm, float* stats,
                              d2s_stream_t stream) {
  D2S_REQUIRE(a && w && x && out_sum, D2S_ERR_ARG, "linear_residual_ln: null pointer");
  D2S_REQUIRE(M >= 0 && (N == 192 || N == 384 || N == 768) && K >= kGpBK && K % kGpBK == 0, D2S_ERR_ARG,
              "linear_residual_ln: need N in {192, 384, 768} (a CTA keeps whole rows: in TMEM, or in two 384-column halves) and "
              "K %% %d == 0 (got M=%d N=%d K=%d)", kGpBK, M, N, K);
  D2S_REQUIRE(!out_norm || (gamma && beta), D2S_ERR_ARG, "linear_residual_ln: out_norm needs gamma and beta");
  D2S_REQUIRE(aligned16(a) && aligned16(w) && aligned16(x) && aligned16(out_sum) && aligned16(out_norm), D2S_ERR_ALIGN,
              "linear_residual_ln: pointers must be 16-byte aligned");
  if (M == 0) return D2S_OK;
  CUtensorMap ma, mw;
  int rc;
  if ((rc = gp_map_2d(&ma, a, K, M, kGpBK, kGpBM, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, what))) return rc;
  if ((rc = gp_map_2d(&mw, w, K, N, kGpBK, 96, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, what))) return rc;
  GpParams p{(const __nv_bfloat16*)bias, (const __nv_bfloat16*)gamma, (const __nv_bfloat16*)beta, (const __nv_bfloat16*)x,
             (__nv_bfloat16*)out_sum, (__nv_bfloat16*)out_norm, nullptr, reinterpret_cast<float2*>(stats), eps, M, N, K, 0,
             (out_norm || stats) ? 1 : 0, gp_trace(), 0, 1, nullptr, nullptr, nullptr};
  if (N != 192) return gp_launch<kGpModeLn, 2, 0>(ma, mw, ma, p, (cudaStream_t)stream, what);      // 384, or 768 as two halves
  return gp_launch<kGpModeLn, 1, 0>(ma, mw, ma, p, (cudaStream_t)stream, what);
}

extern "C" int d2s_linear_residual_ln_bf16(const void* a, const void* w, const void* bias, const void* x, const void* gamma,
                                           const void* beta, float eps, int M, int N, int K, void* out_sum, void* out_norm,
                                           d2s_stream_t stream) {
  return gp_linear_residual("d2s_linear_residual_ln_bf16", a, w, bias, x, gamma, beta, eps, M, N, K, out_sum, out_norm, nullptr, stream);
}

extern "C" int d2s_linear_residual_stats_bf16(const void* a, const void* w, const void* bias, const void* x, float eps, int M, int N,
                                              int K, void* out_sum, float* stats, d2s_stream_t stream) {
  D2S_REQUIRE(stats != nullptr && (reinterpret_cast<uintptr_t>(stats) & 7u) == 0, D2S_ERR_ARG,
              "linear_residual_stats: stats must be a non-null, 8-byte aligned (M,2) f32 buffer");
  return gp_linear_residual("d2s_linear_residual_stats_bf16", a, w, bias, x, nullptr, nullptr, eps, M, N, K, out_sum, nullptr, stats, stream);
}

extern "C" int d2s_linear_act_pair_bf16(const void* a, const void* w, const void* bias, int M, int N, int K, int act, void* out,
                                        void* pre, d2s_stream_t stream) {
  return gp_linear_act("d2s_linear_act_pair_bf16", a, nullptr, nullptr, nullptr, w, bias, M, N, K, act, out, pre, stream);
}

extern "C" int d2s_linear_lnin_act_pair_bf16(const void* x, const float* in_stats, const void* in_gamma, const void* in_beta,
                                             const void* w, const void* bias, int M, int N, int K, int act, void* out,
                                             d2s_stream_t stream) {
  D2S_REQUIRE(in_stats && in_gamma && in_beta && (reinterpret_cast<uintptr_t>(in_stats) & 7u) == 0, D2S_ERR_ARG,
              "linear_lnin_act_pair: in_stats (M,2) f32 (8-byte aligned), in_gamma and in_beta are required");
  return gp_linear_act("d2s_linear_lnin_act_pair_bf16", x, in_stats, in_gamma, in_beta, w, bias, M, N, K, act, out, nullptr, stream);
}
