// Kernel family (1), predictor tail section: the second half of PredictorLG.forward of Variant A
// (vit_models/default_dynamic_vit.py:304-330) fused with the stage's selection (:461-467) as ONE tcgen05 kernel (bf16, D = 384):
//
//   u  = GELU(local @ W2[:, :D/2]^T + (pooled @ W2[:, D/2:]^T + b2))        out_conv[0:2] applied to cat(local, pooled.expand) (:329)
//   v  = GELU(Linear(D/2, D/4)(u))                                          out_conv[2:4]
//   logp = LogSoftmax(Linear(D/4, 2)(v));  kept = argsort(logp[:, :, 0], descending)[:, :K]        out_conv[4:6], :461-465
//
// local (B,N,D/2) = GELU(in_conv)(x)[:, :, :D/2] -- dense from d2s_pool_act, or the first D/2 columns of the (B,N,D) output of the
// Linear + GELU GEMM read in place through the tensor map's row stride --; the per-image term pooled @ W2[:, D/2:]^T + b2 (B,D/2)
// from one small library GEMM over d2s_pool_act's pooled rows.
// Before: two library GEMMs + bias_act + the score-tail kernel (6 launches, (B,N,D/2) written and read twice and (B,N,D/4) once).  Here `local` is read once and only (B,N,2) + (B,K) are written; u and v live in TMEM / shared memory.
//
// One persistent CTA per SM.  W2[:, :D/2] (72 KB) and W3 (36 KB) stay RESIDENT in shared memory (SWIZZLE_128B B operands), so the
// only stream is `local`: 128-row tiles of an image (N <= 256: one or two) through a two-slot ring.  Per tile:
//   G2  acc = tile @ W2l^T (M 128, N 192, K 192)   -> E2: + per-image bias -> GELU -> bf16 IN PLACE over the tile's slot (A operand)
//   G3  acc = u @ W3^T     (M 128, N 96,  K 192)   -> E3: GELU -> two dot products -> log-softmax -> logp out, score key
// and per image the stable descending rank by counting over its N keys (same rule as d2s_select_topk_f32), by two dedicated warps
// while the epilogue warps are already on the next image.  The second Linear's accumulator is double-buffered and the epilogues
// run E2 of the next tile before E3 of this one, so neither product is ever waited for.  The kernel is bound by the epilogues'
// instruction issue (288 exact-erf GELUs per token row), not by HBM or the tensor pipe.
//
//   warps 0-11 epilogues, three per TMEM lane quadrant (row = TMEM lane, each warp a third of the 32-column chunks)
//   warp 12    TMA producer (tiles, resident weights, the image's bias row as a 1-D bulk copy)
//   warp 13    TMEM allocation, tcgen05.mma issue (one elected lane)
//   warps 14-15 selection
//
// Roundings follow the unfused path (and the reference's bf16 modules): every Linear output and every GELU output is rounded to
// bf16; the per-image bias and the last Linear + log-softmax stay in fp32.
//
// The whole predictor as one kernel (first Linear included, in two passes over the image) was built first and measured slower
// than the unfused sequence: W1 has to be re-streamed for every 128-row tile and the per-image dependency chain keeps the
// operand stream, the MMAs and 672 GELUs per row from overlapping (profiles/r02x_predictor_full_fusion.txt).
#include "d2s_tc.cuh"

namespace d2s {

constexpr int kPfH = 192, kPfQ = 96;                    // D/2, D/4
constexpr int kPfMaxN = 256;
constexpr int kPfParts = 3;                             // epilogue warps per TMEM lane quadrant
constexpr int kPfEThreads = 128 * kPfParts;
constexpr int kPfSelWarps = 2;
constexpr int kPfThreads = kPfEThreads + 64 + 32 * kPfSelWarps;   // + TMA producer warp + MMA warp + selection warps
constexpr int kPfTmaWarp = 4 * kPfParts, kPfMmaWarp = 4 * kPfParts + 1, kPfSelWarp0 = 4 * kPfParts + 2;
constexpr uint32_t kPfABytes = 128 * 128;               // 128 rows x 64 bf16
constexpr uint32_t kPfW2Bytes = 192 * 128;              // 192 rows x 64 bf16
constexpr uint32_t kPfW3Bytes = 96 * 128;
constexpr uint32_t kPfSlot = 3 * kPfABytes;             // one 128 x 192 bf16 tile as three 64-column blocks
constexpr uint32_t kPfAccB = 0, kPfAccC = 384;          // TMEM columns: second Linear (2 x 192), third Linear (96)

struct PfBars {
  uint64_t w_full, a_full[2], a_empty[2], b_full[2], b_empty[2], c_full, c_empty, u_full[2];
  uint64_t pi_full[2], pi_empty[2], key_full[2], key_empty[2];
  uint32_t tmem_base;
  uint32_t pad;
};

struct PfSmall {                       // behind the resident weights and the tile slots
  PfBars bars;
  alignas(16) float b3[kPfQ];
  alignas(16) float w4[2 * kPfQ];
  alignas(16) __nv_bfloat16 per_image[2][kPfH];   // the image's bias of the second Linear (double-buffered over images)
  alignas(16) float2 dot[3][128];                 // last Linear: partial dot products per 32-column chunk of the third Linear
  alignas(16) uint32_t key[2][kPfMaxN + 4];       // score keys of an image (double-buffered: selection runs under the next image)
};

struct PfParams {
  const __nv_bfloat16 *per_image, *b3;
  const float *w4, *b4, *prev;
  float* logp;
  int64_t* kept;
  float* prev_kept;
  int B, N, K;
};

// bf16(GELU(bf16(x))) for a pair, as the separate Linear -> GELU modules round
__device__ __forceinline__ uint32_t pf_gelu_bf16(float x0, float x1) {
  const uint32_t zb = pack_bf16x2(x0, x1);
  float g0, g1;
  f2_unpack(gelu_erf_pair(f2_pack(bf16_lo(zb), bf16_hi(zb))), g0, g1);
  return pack_bf16x2(g0, g1);
}

__global__ void __launch_bounds__(kPfThreads, 1)
predictor_a_tail_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w2,
                        const __grid_constant__ CUtensorMap map_w3, const PfParams p) {
  extern __shared__ unsigned char smem_dyn[];
  const uint32_t raw = smem_u32(smem_dyn);
  const uint32_t padb = (1024u - (raw & 1023u)) & 1023u;
  unsigned char* w2_s = smem_dyn + padb;                  // 3 x [192 rows x 128 B]
  unsigned char* w3_s = w2_s + 3 * kPfW2Bytes;            // 3 x [96 rows x 128 B]
  unsigned char* slots = w3_s + 3 * kPfW3Bytes;           // 2 x 3 x [128 rows x 128 B]
  PfSmall* sm = reinterpret_cast<PfSmall*>(slots + 2 * kPfSlot);
  PfBars* bars = &sm->bars;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.N, nt = (N + 127) >> 7;
  const int my_imgs = p.B > (int)blockIdx.x ? (p.B - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  const int units = my_imgs * nt;                         // (image, tile) units of this CTA, in order

  if (tid == 0) {
    mbar_init(smem_u32(&bars->w_full), 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&bars->a_full[i]), 1);
      mbar_init(smem_u32(&bars->a_empty[i]), 1);
      mbar_init(smem_u32(&bars->b_full[i]), 1);
      mbar_init(smem_u32(&bars->b_empty[i]), kPfEThreads);
      mbar_init(smem_u32(&bars->u_full[i]), kPfEThreads);
      mbar_init(smem_u32(&bars->pi_full[i]), 1);
      mbar_init(smem_u32(&bars->pi_empty[i]), kPfEThreads);
      mbar_init(smem_u32(&bars->key_full[i]), kPfEThreads);
      mbar_init(smem_u32(&bars->key_empty[i]), kPfSelWarps);
    }
    mbar_init(smem_u32(&bars->c_full), 1);
    mbar_init(smem_u32(&bars->c_empty), kPfEThreads);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kPfMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  for (int i = tid; i < 2 * kPfQ; i += kPfThreads) sm->w4[i] = p.w4[i];
  for (int i = tid; i < kPfQ; i += kPfThreads) sm->b3[i] = __bfloat162float(p.b3[i]);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;

  if (warp == kPfTmaWarp) {
    if (lane == 0) {
      // ================================================ TMA producer ================================================
      const uint32_t wf = smem_u32(&bars->w_full);
      mbar_expect_tx(wf, 3 * kPfW2Bytes + 3 * kPfW3Bytes);
      for (int kb = 0; kb < 3; ++kb) {
        tma_load_2d(smem_u32(w2_s + kb * kPfW2Bytes), &map_w2, kb * 64, 0, wf);
        tma_load_2d(smem_u32(w3_s + kb * kPfW3Bytes), &map_w3, kb * 64, 0, wf);
      }
      for (int u = 0; u < units; ++u) {
        const int i = u / nt, t = u - i * nt;
        const int img = (int)blockIdx.x + i * (int)gridDim.x;
        if (t == 0) {                                        // the image's bias row of the second Linear: one 384-byte bulk copy
          const uint32_t pb = i & 1;
          mbar_wait(smem_u32(&bars->pi_empty[pb]), ((i >> 1) & 1) ^ 1);
          const uint32_t pf = smem_u32(&bars->pi_full[pb]);
          mbar_expect_tx(pf, kPfH * 2);
          bulk_load_1d(smem_u32(&sm->per_image[pb][0]), p.per_image + (size_t)img * kPfH, kPfH * 2, pf);
        }
        const uint32_t s = u & 1, n = u >> 1;
        mbar_wait(smem_u32(&bars->a_empty[s]), (n & 1) ^ 1);
        const uint32_t full = smem_u32(&bars->a_full[s]);
        mbar_expect_tx(full, kPfSlot);
        for (int kb = 0; kb < 3; ++kb) tma_load_3d(smem_u32(slots + s * kPfSlot + kb * kPfABytes), &map_x, kb * 64, t * 128, img, full);
      }
    }
  } else if (warp_uniform(warp) == kPfMmaWarp) {
    // ===== MMA issuer: the whole warp runs the loop warp-uniformly, one elected lane issues (see elect_one, d2s_tc.cuh) =====
    const uint32_t idesc_h = make_idesc(128, kPfH, 0), idesc_q = make_idesc(128, kPfQ, 0);
    mbar_wait(smem_u32(&bars->w_full), 0);
    auto g2 = [&](int u) {                                   // second Linear of unit u
      const uint32_t s = u & 1, n = u >> 1;
      mbar_wait(smem_u32(&bars->a_full[s]), n & 1);
      mbar_wait(smem_u32(&bars->b_empty[s]), (n & 1) ^ 1);
      tc_fence_after();
      const uint32_t d = tmem + kPfAccB + s * kPfH;
#pragma unroll
      for (int kb = 0; kb < 3; ++kb) {
        const uint64_t ad = make_desc_sw128(smem_u32(slots + s * kPfSlot + kb * kPfABytes), 16, 1024);
        const uint64_t bd = make_desc_sw128(smem_u32(w2_s + kb * kPfW2Bytes), 16, 1024);
        if (elect_one()) {
          if (kb == 0) mma_ss_imm<false>(d, ad, bd, idesc_h); else mma_ss_imm<true>(d, ad, bd, idesc_h);
          mma_ss_imm<true>(d, ad + 2, bd + 2, idesc_h);
          mma_ss_imm<true>(d, ad + 4, bd + 4, idesc_h);
          mma_ss_imm<true>(d, ad + 6, bd + 6, idesc_h);
        }
        __syncwarp();
      }
      if (elect_one()) mma_commit(smem_u32(&bars->b_full[s]));
      __syncwarp();
    };
    auto g3 = [&](int u) {                                   // third Linear of unit u: A = u written in place over the tile
      const uint32_t s = u & 1, n = u >> 1;
      mbar_wait(smem_u32(&bars->u_full[s]), n & 1);
      mbar_wait(smem_u32(&bars->c_empty), (u & 1) ^ 1);
      tc_fence_after();
      const uint32_t d = tmem + kPfAccC;
#pragma unroll
      for (int kb = 0; kb < 3; ++kb) {
        const uint64_t ad = make_desc_sw128(smem_u32(slots + s * kPfSlot + kb * kPfABytes), 16, 1024);
        const uint64_t bd = make_desc_sw128(smem_u32(w3_s + kb * kPfW3Bytes), 16, 1024);
        if (elect_one()) {
          if (kb == 0) mma_ss_imm<false>(d, ad, bd, idesc_q); else mma_ss_imm<true>(d, ad, bd, idesc_q);
          mma_ss_imm<true>(d, ad + 2, bd + 2, idesc_q);
          mma_ss_imm<true>(d, ad + 4, bd + 4, idesc_q);
          mma_ss_imm<true>(d, ad + 6, bd + 6, idesc_q);
        }
        __syncwarp();
      }
      if (elect_one()) {
        mma_commit(smem_u32(&bars->c_full));
        mma_commit(smem_u32(&bars->a_empty[s]));             // the slot may be refilled once these MMAs have read it
      }
      __syncwarp();
    };
    if (units > 0) g2(0);
    for (int u = 0; u < units; ++u) {
      if (u + 1 < units) g2(u + 1);                          // runs under E2 / E3 of unit u
      g3(u);
    }
  } else if (warp >= kPfSelWarp0) {
    // ===== selection warps: stable descending rank by counting (d2s_select.cu) over an image's keys, while the epilogue
    // warps are already on the next image.  Warp w takes tokens w*32 + lane + 64 j. =====
    const int sw = warp - kPfSelWarp0;
    for (int i = 0; i < my_imgs; ++i) {
      const int img = (int)blockIdx.x + i * (int)gridDim.x;
      const uint32_t kb = i & 1;
      mbar_wait(smem_u32(&bars->key_full[kb]), (i >> 1) & 1);
      const float* prev_b = p.prev ? p.prev + (size_t)img * N : nullptr;
      const uint4* k4 = reinterpret_cast<const uint4*>(sm->key[kb]);
      const int n4 = (N + 3) >> 2;
      constexpr int kTok = kPfMaxN / (32 * kPfSelWarps);
      uint32_t my[kTok];
      int rk[kTok];
#pragma unroll
      for (int j = 0; j < kTok; ++j) {
        const int tok = sw * 32 + lane + 32 * kPfSelWarps * j;
        my[j] = tok < N ? sm->key[kb][tok] : 0u;
        rk[j] = 0;
      }
#pragma unroll 2
      for (int j4 = 0; j4 < n4; ++j4) {
        const uint4 k = k4[j4];
        const int jj = 4 * j4;
#pragma unroll
        for (int j = 0; j < kTok; ++j) {
          const int tok = sw * 32 + lane + 32 * kPfSelWarps * j;
          rk[j] += (int)((k.x > my[j]) || (k.x == my[j] && jj < tok)) + (int)((k.y > my[j]) || (k.y == my[j] && jj + 1 < tok)) +
                   (int)((k.z > my[j]) || (k.z == my[j] && jj + 2 < tok)) + (int)((k.w > my[j]) || (k.w == my[j] && jj + 3 < tok));
        }
      }
#pragma unroll
      for (int j = 0; j < kTok; ++j) {
        const int tok = sw * 32 + lane + 32 * kPfSelWarps * j;
        if (tok < N && rk[j] < p.K) {
          p.kept[(size_t)img * p.K + rk[j]] = tok;
          if (p.prev_kept) p.prev_kept[(size_t)img * p.K + rk[j]] = prev_b ? prev_b[tok] : 1.0f;
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&bars->key_empty[kb]));
    }
  } else {
    // ================================================= epilogue warps =================================================
    // warp (quad, part) owns the 32-column chunks c = part, part + kPfParts, ... of every accumulator for the quadrant's 32 rows.
    // E2 of unit u + 1 runs before E3 of unit u, so the third Linear's MMAs are never waited for.
    const int quad = warp & 3, part = warp >> 2;
    const int r = quad * 32 + lane;                               // row inside the tile == TMEM lane
    const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16);
    const float b40 = p.b4[0], b41 = p.b4[1];
    for (int step = 0; step <= units; ++step) {
      if (step < units) {
        // ---- E2: second Linear + per-image bias -> GELU -> u, in place over the tile (A operand of the third Linear) ----
        const int u = step, i = u / nt, t = u - i * nt;
        const uint32_t s = u & 1, ph = (u >> 1) & 1, pb = i & 1;
        const bool quad_active = t * 128 + quad * 32 < N;   // rows past N: nothing to compute (their u rows stay stale)
        if (t == 0) mbar_wait(smem_u32(&bars->pi_full[pb]), (i >> 1) & 1);
        mbar_wait(smem_u32(&bars->b_full[s]), ph);
        tc_fence_after();
        if (quad_active) {
          unsigned char* slot = slots + s * kPfSlot;
          const uint32_t* bias2 = reinterpret_cast<const uint32_t*>(sm->per_image[pb]);
#pragma unroll 1
          for (int c = part; c < 6; c += kPfParts) {
            uint32_t v[32];
            tmem_ld32_nowait(lane_addr + kPfAccB + s * kPfH + c * 32, v);
            tmem_ld_wait();
            uint32_t o[16];
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              const uint4 bw = *reinterpret_cast<const uint4*>(&bias2[c * 16 + 4 * q4]);
              const uint32_t bq[4] = {bw.x, bw.y, bw.z, bw.w};
#pragma unroll
              for (int qq = 0; qq < 4; ++qq) {
                const int q = 4 * q4 + qq;
                o[q] = pf_gelu_bf16(__uint_as_float(v[2 * q]) + bf16_lo(bq[qq]), __uint_as_float(v[2 * q + 1]) + bf16_hi(bq[qq]));
              }
            }
            unsigned char* blk = slot + (c >> 1) * kPfABytes;
#pragma unroll
            for (int q = 0; q < 4; ++q)
              *reinterpret_cast<uint4*>(blk + sw128_off(r, (c & 1) * 4 + q)) = make_uint4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        tc_fence_before();
        mbar_arrive(smem_u32(&bars->b_empty[s]));
        mbar_arrive(smem_u32(&bars->u_full[s]));
        if (t == nt - 1) mbar_arrive(smem_u32(&bars->pi_empty[pb]));
      }
      if (step >= 1) {
        // ---- E3: third Linear -> GELU -> Linear(D/4, 2): partial dot products per 32-column chunk, summed in chunk order ----
        const int u = step - 1, i = u / nt, t = u - i * nt;
        const int img = (int)blockIdx.x + i * (int)gridDim.x;
        const uint32_t kb = i & 1;
        const int n = t * 128 + r;
        const bool quad_active = t * 128 + quad * 32 < N;
        if (t == 0) mbar_wait(smem_u32(&bars->key_empty[kb]), ((i >> 1) & 1) ^ 1);
        mbar_wait(smem_u32(&bars->c_full), u & 1);
        tc_fence_after();
        if (quad_active) {
          for (int c = part; c < 3; c += kPfParts) {
            float a0 = 0.f, a1 = 0.f;
            uint32_t v[32];
            tmem_ld32_nowait(lane_addr + kPfAccC + c * 32, v);
            tmem_ld_wait();
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              const int col = c * 32 + 2 * q;
              const float2 bq = *reinterpret_cast<const float2*>(&sm->b3[col]);
              const uint32_t gb = pf_gelu_bf16(__uint_as_float(v[2 * q]) + bq.x, __uint_as_float(v[2 * q + 1]) + bq.y);
              const float2 w0 = *reinterpret_cast<const float2*>(&sm->w4[col]);
              const float2 w1 = *reinterpret_cast<const float2*>(&sm->w4[kPfQ + col]);
              a0 = fmaf(bf16_lo(gb), w0.x, a0); a0 = fmaf(bf16_hi(gb), w0.y, a0);
              a1 = fmaf(bf16_lo(gb), w1.x, a1); a1 = fmaf(bf16_hi(gb), w1.y, a1);
            }
            sm->dot[c][r] = make_float2(a0, a1);
          }
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&bars->c_empty));
        asm volatile("bar.sync %0, %1;" ::"r"(2 + quad), "n"(32 * kPfParts) : "memory");     // the warps of this lane quadrant
        if (part == 0 && n < N) {
          const float2 d0 = sm->dot[0][r], d1 = sm->dot[1][r], d2 = sm->dot[2][r];
          const float a0 = ((d0.x + d1.x) + d2.x) + b40, a1 = ((d0.y + d1.y) + d2.y) + b41;
          const float m = fmaxf(a0, a1);
          const float lse = m + logf(expf(a0 - m) + expf(a1 - m));
          const float lp0 = a0 - lse, lp1 = a1 - lse;
          reinterpret_cast<float2*>(p.logp)[(size_t)img * N + n] = make_float2(lp0, lp1);
          sm->key[kb][n] = float_to_ordered(lp0);
        }
        if (t == nt - 1 && tid < 4) sm->key[kb][N + tid] = 0u;   // padding of the 4-wide rank loop: below every real key
        asm volatile("bar.sync %0, %1;" ::"r"(2 + quad), "n"(32 * kPfParts) : "memory");     // dot[] is rewritten by the next tile
        if (t == nt - 1) mbar_arrive(smem_u32(&bars->key_full[kb]));                          // (release: the keys above are visible)
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kPfMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512) : "memory");
  }
}

static int pf_map(CUtensorMap* map, const void* base, int rank, const cuuint64_t* gdim, const cuuint64_t* gstr,
                  const cuuint32_t* box, CUtensorMapL2promotion promo, const char* what) {
  GgEncodeFn enc = gg_encode_fn();
  D2S_REQUIRE(enc != nullptr, D2S_ERR_CUDA, "%s: cuTensorMapEncodeTiled is unavailable from the driver", what);
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult cr = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  D2S_REQUIRE(cr == CUDA_SUCCESS, D2S_ERR_CUDA, "%s: tensor map encode failed (%d)", what, (int)cr);
  return D2S_OK;
}

}  // namespace d2s

using namespace d2s;

extern "C" int d2s_predictor_a_tail_bf16(const void* local, int ld, long long lb, const void* per_image, const void* w2, const void* w3,
                                         const void* b3, const float* w4, const float* b4, const float* prev, int B, int N, int H,
                                         int K, float* logp, int64_t* kept, float* prev_kept, d2s_stream_t stream) {
  const char* what = "d2s_predictor_a_tail_bf16";
  D2S_REQUIRE(local && per_image && w2 && w3 && b3 && w4 && b4 && logp && (kept || K == 0), D2S_ERR_ARG, "predictor_a_tail: null pointer");
  D2S_REQUIRE(H == kPfH, D2S_ERR_ARG, "predictor_a_tail: H=%d unsupported (the kernel is built for D/2 = %d)", H, kPfH);
  D2S_REQUIRE(B >= 0 && N >= 1 && N <= kPfMaxN, D2S_ERR_ARG, "predictor_a_tail: N=%d outside [1,%d]", N, kPfMaxN);
  D2S_REQUIRE(K >= 0 && K <= N, D2S_ERR_ARG, "predictor_a_tail: K=%d outside [0,N=%d]", K, N);
  D2S_REQUIRE(ld >= H && ld % 8 == 0, D2S_ERR_ARG, "predictor_a_tail: row stride ld=%d must be a multiple of 8 elements, at least H=%d", ld, H);
  D2S_REQUIRE(lb >= (long long)N * ld && lb % 8 == 0, D2S_ERR_ARG,
              "predictor_a_tail: batch stride lb=%lld must be a multiple of 8 elements, at least N * ld", lb);
  D2S_REQUIRE(aligned16(local) && aligned16(per_image) && aligned16(w2) && aligned16(w3) && aligned16(logp), D2S_ERR_ALIGN,
              "predictor_a_tail: local / per_image / weights / logp must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  CUtensorMap mx, mw2, mw3;
  int rc;
  {
    const cuuint64_t gdim[3] = {(cuuint64_t)H, (cuuint64_t)N, (cuuint64_t)B};
    const cuuint64_t gstr[2] = {(cuuint64_t)ld * 2, (cuuint64_t)lb * 2};
    const cuuint32_t box[3] = {64, 128, 1};
    if ((rc = pf_map(&mx, local, 3, gdim, gstr, box, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, what))) return rc;
  }
  {
    const cuuint64_t gdim[2] = {(cuuint64_t)2 * H, (cuuint64_t)H};
    const cuuint64_t gstr[1] = {(cuuint64_t)2 * H * 2};
    const cuuint32_t box[2] = {64, (cuuint32_t)kPfH};
    if ((rc = pf_map(&mw2, w2, 2, gdim, gstr, box, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, what))) return rc;
  }
  {
    const cuuint64_t gdim[2] = {(cuuint64_t)H, (cuuint64_t)kPfQ};
    const cuuint64_t gstr[1] = {(cuuint64_t)H * 2};
    const cuuint32_t box[2] = {64, (cuuint32_t)kPfQ};
    if ((rc = pf_map(&mw3, w3, 2, gdim, gstr, box, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, what))) return rc;
  }
  PfParams p{(const __nv_bfloat16*)per_image, (const __nv_bfloat16*)b3, w4, b4, prev, logp, kept, prev_kept, B, N, K};
  const size_t smem = 1024 + (size_t)3 * kPfW2Bytes + 3 * kPfW3Bytes + 2 * kPfSlot + sizeof(PfSmall);
  D2S_REQUIRE(smem <= 227 * 1024, D2S_ERR_ARG, "%s: needs %zu B of shared memory", what, smem);
  static SmemOptIn opt;
  cudaError_t e = opt_in_smem(opt, predictor_a_tail_kernel, 227 * 1024);
  D2S_REQUIRE(e == cudaSuccess, D2S_ERR_CUDA, "%s: cudaFuncSetAttribute: %s", what, cudaGetErrorString(e));
  const int grid = B < kNumSMs ? B : kNumSMs;
  predictor_a_tail_kernel<<<grid, kPfThreads, smem, (cudaStream_t)stream>>>(mx, mw2, mw3, p);
  count_launch();
  return check_launch(what);
}
