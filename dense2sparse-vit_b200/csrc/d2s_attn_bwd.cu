// Kernel family (4), training form: backward of the policy-masked attention on tcgen05 / TMEM (bf16 in, fp32 accumulate).
// No (B,H,T,T) tensor exists anywhere: scores and probabilities are recomputed from the packed qkv and the per-row statistics
// the forward saved (d2s_attn_policy_fwd, `stats`), as in flash attention, and the keep-policy gradient falls out of the
// same pass.  Reference: Attention.softmax_with_policy + Attention.forward under autograd
// (vit_models/dynamic_vit.py:195-236 == default_dynamic_vit.py:185-216).
//
//   forward (per image b, head h; z = scale * q k^T, k2 = scale * log2 e):
//     e~_ij = 2^(k2 s_ij - m'_i)          m_ij = p_j + (1 - p_j) [i == j]          e_ij = e~_ij m_ij
//     P_ij  = (e_ij + c_i) / den_i         den_i = sum_j e_ij + eps'_i,  c_i = eps'_i / T          O = P V
//   backward, given dO (and optionally g_cls = d loss / d P[0, :]):
//     dP = dO V^T (+ g_cls on row 0)       delta_i = sum_j dP_ij P_ij = dO_i . O_i (+ g_cls . P_0)
//     g_ij = (dP_ij - delta_i) / den_i     dS_ij = g_ij e_ij                        d p_j = sum_h sum_{i != j} g_ij e~_ij
//     dV = P^T dO        dK = scale dS^T Q        dQ = scale dS K
//   (the gradient through the subtracted row maximum is O(eps) -- see d2s_attn_simt.cu -- and is dropped, as in the padded-row
//   bf16 kernels this replaces.)
//
// Orientation.  The tile is TRANSPOSED with respect to the forward kernel: TMEM lanes are KEYS, columns are queries,
//     S^T = K_jb Q^T     dP^T = V_jb dO^T          (SS MMAs, M = 128 keys of key tile jb, N = Tp queries, K = 64)
// so that (a) P^T and dS^T, written back over the consumed columns as packed bf16, are directly the TMEM A operands of
//     dV_jb = P^T dO     dK_jb = dS^T Q            (TS MMAs, B = dO / Q read MN-major from the same shared-memory tiles)
// with no reduction across tiles, and (b) the policy gradient of key j is a plain per-thread sum over the row.  The per-query
// statistics (m', 1/den, -delta/den, c/den) are shared-memory broadcasts.  Only dQ needs dS with queries as rows: every thread
// also writes its dS^T row into a SWIZZLE_128B shared-memory tile laid out [64-query block][key row][128 B], which is at the
// same time the canonical MN-major A operand (M = queries) of
//     dQ_t += dS K_jb                               (SS MMA, A MN-major, B = K_jb MN-major)
// dQ is accumulated over the two key tiles through a small fp32 stash in shared memory (T > 128 only).
//
// TMEM (512 columns): S^T [0, 208) -> P^T [0, 104) + dV_jb [104, 168);  dP^T [208, 416) -> dS^T [208, 312) + dK_jb [312, 376);
// dQ_t [416, 480).  One persistent CTA per SM; warps 0-3 = one key row per thread (TMEM lane quadrant = warp), warp 4 issues TMA
// and MMAs.  Per (image, head): 24.8 MFLOP against 8 x T x 64 x 2 B = 202 KB of HBM traffic at T = 197 -- HBM-bound, like the
// forward.
#include "d2s_tc.cuh"

namespace d2s {

constexpr int kBwdMaxT = 208;                 // S^T + dP^T + dQ_t must fit 512 TMEM columns
constexpr uint32_t kColS = 0, kColDP = 208, kColDV = 104, kColDK = 312, kColDQ = 416;
constexpr int kBwdThreads = 160;

struct BwdBars {
  uint64_t qdo_full, k_full[2], v_full, sdp_full, pds_full, acc_full, acc_free, dq_full, dq_free;
  uint32_t tmem_base;
  uint32_t pad;
};

// delta_i = dO_i . O_i (+ g_cls . cls_row for query 0), stored in stats[..][3].  8 lanes per (token, head) row of 64 bf16.
__global__ void __launch_bounds__(256)
attn_bwd_prep_kernel(const __nv_bfloat16* __restrict__ O, const __nv_bfloat16* __restrict__ dO,
                     const float* __restrict__ cls_row, const float* __restrict__ g_cls, long long rows, int T, int H,
                     float* __restrict__ stats) {
  const int sub = threadIdx.x & 7;
  const long long row = (long long)blockIdx.x * 32 + (threadIdx.x >> 3);      // (b * T + i) * H + h
  if (row >= rows) return;                                                    // (whole 8-lane groups leave together)
  const uint4 a = ld_nc16(O + row * 64 + sub * 8), g = ld_nc16(dO + row * 64 + sub * 8);
  float acc = bf16_lo(a.x) * bf16_lo(g.x) + bf16_hi(a.x) * bf16_hi(g.x) + bf16_lo(a.y) * bf16_lo(g.y) + bf16_hi(a.y) * bf16_hi(g.y) +
              bf16_lo(a.z) * bf16_lo(g.z) + bf16_hi(a.z) * bf16_hi(g.z) + bf16_lo(a.w) * bf16_lo(g.w) + bf16_hi(a.w) * bf16_hi(g.w);
  const int h = (int)(row % H);
  const long long bt = row / H;
  const int i = (int)(bt % T);
  const long long b = bt / T;
  const size_t unit = (size_t)b * H + h;
  if (g_cls != nullptr && i == 0)
    for (int j = sub; j < T; j += 8) acc += g_cls[unit * T + j] * cls_row[unit * T + j];
  const unsigned gm = 0xffu << (threadIdx.x & 24);
  acc += __shfl_xor_sync(gm, acc, 1);
  acc += __shfl_xor_sync(gm, acc, 2);
  acc += __shfl_xor_sync(gm, acc, 4);
  if (sub == 0) stats[(unit * T + i) * 4 + 3] = acc;
}

// kNT  : 128-row tiles per unit, keys and queries alike (1: T <= 128, 2: T <= 208)
// kPol : keep policy given (masked exponentials, d policy)
template <int kNT, bool kPol>
__global__ void __launch_bounds__(kBwdThreads, 1)
attn_tc_bwd_kernel(const __grid_constant__ CUtensorMap map_qa, const __grid_constant__ CUtensorMap map_qb,
                   const __grid_constant__ CUtensorMap map_ga, const __grid_constant__ CUtensorMap map_gb,
                   const float* __restrict__ policy, const float* __restrict__ stats, const float* __restrict__ g_cls,
                   int num_units, int T, int H, int Tp, float scale, __nv_bfloat16* __restrict__ dqkv,
                   float* __restrict__ gpolicy) {
  extern __shared__ unsigned char smem_dyn[];
  const uint32_t raw = smem_u32(smem_dyn);
  const uint32_t pad = (1024u - (raw & 1023u)) & 1023u;
  unsigned char* tiles = smem_dyn + pad;
  const int rows_a = kNT == 1 ? Tp : kTileRows;          // rows of the first TMA box, and of key tile 0
  const int rows_b = kNT == 1 ? 0 : Tp - kTileRows;      // rows of the second box, and of key tile 1
  unsigned char* q_s = tiles;                                      // Tp x 128 B (Tp is a multiple of 16: whole 1024-byte atoms)
  unsigned char* do_s = q_s + (size_t)Tp * 128;                    // Tp x 128 B
  unsigned char* k_s = do_s + (size_t)Tp * 128;                    // 2 x 128 x 128 B  (key tile jb; double-buffered: K lives until the dQ MMAs)
  unsigned char* v_s = k_s + 2 * kTileBytes;                       // 128 x 128 B
  unsigned char* ds_s = v_s + kTileBytes;                          // 2 kNT blocks of [128 key rows x 64 queries]: dS^T
  float* stash = reinterpret_cast<float*>(ds_s + (size_t)2 * kNT * kTileBytes);   // kNT == 2: Tp x 64 fp32 (dQ of key tile 0)
  // per-query statistics, two queries per entry for the packed fp32x2 arithmetic of the pass:
  //   sts[2 p] = (-m'_i, -m'_i+1, 1/den_i, 1/den_i+1)      sts[2 p + 1] = (-delta_i/den_i, -delta_i+1/den_i+1, c_i/den_i, c_i+1/den_i+1),  i = 2 p
  float4* sts = reinterpret_cast<float4*>(stash + (kNT == 2 ? (size_t)Tp * kTcHD : 0));   // 256 floats x 4
  float* pol_s = reinterpret_cast<float*>(sts + 256);              // 256
  BwdBars* bars = reinterpret_cast<BwdBars*>(pol_s + 256);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    mbar_init(smem_u32(&bars->qdo_full), 1);
    mbar_init(smem_u32(&bars->k_full[0]), 1);
    mbar_init(smem_u32(&bars->k_full[1]), 1);
    mbar_init(smem_u32(&bars->v_full), 1);
    mbar_init(smem_u32(&bars->sdp_full), 1);
    mbar_init(smem_u32(&bars->pds_full), 128);
    mbar_init(smem_u32(&bars->acc_full), 1);
    mbar_init(smem_u32(&bars->acc_free), 128);
    mbar_init(smem_u32(&bars->dq_full), 1);
    mbar_init(smem_u32(&bars->dq_free), 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)), "n"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;
  const int nchunks = Tp / 16;

  if (warp_uniform(warp) == 4) {
    // =============================== control warp: TMA + MMA issue (warp-uniform, one elected lane) ===============================
    const uint32_t idesc_s = make_idesc(128, Tp, 0);            // S^T, dP^T: N = queries
    const uint32_t idesc_kv = make_idesc(128, kTcHD, 1);        // dV, dK: A from TMEM, B MN-major
    const uint32_t idesc_q = make_idesc(128, kTcHD, 1, 1);      // dQ: A and B MN-major
    const uint64_t qd = make_desc_sw128(smem_u32(q_s), 16, 1024), gd = make_desc_sw128(smem_u32(do_s), 16, 1024);
    const uint64_t kd0 = make_desc_sw128(smem_u32(k_s), 16, 1024), vd = make_desc_sw128(smem_u32(v_s), 16, 1024);
    const uint32_t bytes_a = (uint32_t)rows_a * 128u, bytes_b = (uint32_t)rows_b * 128u;
    auto load_qdo = [&](int unit) {     // all Tp query rows of Q and dO
      const uint32_t bar = smem_u32(&bars->qdo_full);
      if (elect_one()) {
        mbar_expect_tx(bar, 2 * (bytes_a + bytes_b));
        const int b = unit / H, h = unit % H;
        tma_load_3d(smem_u32(q_s), &map_qa, h * kTcHD, 0, b, bar);
        tma_load_3d(smem_u32(do_s), &map_ga, h * kTcHD, 0, b, bar);
        if (kNT == 2) {
          tma_load_3d(smem_u32(q_s) + bytes_a, &map_qb, h * kTcHD, kTileRows, b, bar);
          tma_load_3d(smem_u32(do_s) + bytes_a, &map_gb, h * kTcHD, kTileRows, b, bar);
        }
      }
      __syncwarp();
    };
    auto load_tile = [&](unsigned char* dst, int which, int unit, int jb, uint32_t bar) {   // key tile jb of K (1) or V (2)
      if (elect_one()) {
        mbar_expect_tx(bar, jb == 0 ? bytes_a : bytes_b);
        tma_load_3d(smem_u32(dst), jb == 0 ? &map_qa : &map_qb, (which * H + unit % H) * kTcHD, jb * kTileRows, unit / H, bar);
      }
      __syncwarp();
    };
    int unit = blockIdx.x;
    if (unit < num_units) {
      load_qdo(unit);
      load_tile(k_s, 1, unit, 0, smem_u32(&bars->k_full[0]));
      load_tile(v_s, 2, unit, 0, smem_u32(&bars->v_full));
    }
    uint32_t iter = 0, dqn = 0, un = 0;     // (unit, key tile) iterations, dQ tiles and units processed by this CTA: parity sources
    for (; unit < num_units; unit += gridDim.x, ++un) {
      const int next = unit + gridDim.x;
#pragma unroll
      for (int jb = 0; jb < kNT; ++jb, ++iter) {
        const bool last_jb = jb == kNT - 1;
        const int n_unit = last_jb ? next : unit, n_jb = last_jb ? 0 : jb + 1;     // the (unit, key tile) after this one
        const bool has_n = n_unit < num_units;
        const uint32_t kb = iter & 1;                                              // K buffer of this iteration
        const uint64_t kd = kd0 + (uint64_t)(kb * (kTileBytes >> 4));
        if (has_n) {
          // the other K buffer was last read by the dQ MMAs of the previous iteration: refill it a whole iteration ahead
          if (iter > 0) mbar_wait(smem_u32(&bars->dq_full), (dqn - 1) & 1);
          load_tile(k_s + (kb ^ 1) * kTileBytes, 1, n_unit, n_jb, smem_u32(&bars->k_full[kb ^ 1]));
        }
        if (jb == 0) mbar_wait(smem_u32(&bars->qdo_full), un & 1);
        mbar_wait(smem_u32(&bars->k_full[kb]), (iter >> 1) & 1);
        mbar_wait(smem_u32(&bars->v_full), iter & 1);
        if (iter > 0) mbar_wait(smem_u32(&bars->acc_free), (iter - 1) & 1);        // dV / dK of the previous tile are drained
        tc_fence_after();
        if (elect_one()) {
          mma_ss_imm<false>(tmem + kColS, kd, qd, idesc_s);
          mma_ss_imm<true>(tmem + kColS, kd + 2, qd + 2, idesc_s);
          mma_ss_imm<true>(tmem + kColS, kd + 4, qd + 4, idesc_s);
          mma_ss_imm<true>(tmem + kColS, kd + 6, qd + 6, idesc_s);
          mma_ss_imm<false>(tmem + kColDP, vd, gd, idesc_s);
          mma_ss_imm<true>(tmem + kColDP, vd + 2, gd + 2, idesc_s);
          mma_ss_imm<true>(tmem + kColDP, vd + 4, gd + 4, idesc_s);
          mma_ss_imm<true>(tmem + kColDP, vd + 6, gd + 6, idesc_s);
          mma_commit(smem_u32(&bars->sdp_full));
        }
        __syncwarp();
        mbar_wait(smem_u32(&bars->sdp_full), iter & 1);                            // V tile is dead: fetch the next one
        if (has_n) load_tile(v_s, 2, n_unit, n_jb, smem_u32(&bars->v_full));
        mbar_wait(smem_u32(&bars->pds_full), iter & 1);                            // P^T, dS^T in TMEM; dS in shared memory
        tc_fence_after();
        if (elect_one()) {
          mma_ts_imm<false>(tmem + kColDV, tmem + kColS, gd, idesc_kv);
#pragma unroll
          for (int ks = 1; ks < kBwdMaxT / 16; ++ks)
            if (ks < nchunks) mma_ts_imm<true>(tmem + kColDV, tmem + kColS + ks * 8, gd + (uint64_t)(ks * 128), idesc_kv);
          mma_ts_imm<false>(tmem + kColDK, tmem + kColDP, qd, idesc_kv);
#pragma unroll
          for (int ks = 1; ks < kBwdMaxT / 16; ++ks)
            if (ks < nchunks) mma_ts_imm<true>(tmem + kColDK, tmem + kColDP + ks * 8, qd + (uint64_t)(ks * 128), idesc_kv);
          mma_commit(smem_u32(&bars->acc_full));
        }
        __syncwarp();
        const int ksteps = (jb == 0 ? rows_a : rows_b) / 16;                       // key rows of this tile / 16
#pragma unroll
        for (int t = 0; t < kNT; ++t, ++dqn) {
          if (dqn > 0) mbar_wait(smem_u32(&bars->dq_free), (dqn - 1) & 1);         // previous dQ tile is drained
          tc_fence_after();
          // A = dS, M = queries [128 t, 128 t + 128): two 64-query blocks 16 KB apart (LBO), 8 key rows per 1024 B (SBO)
          const uint64_t ad = make_desc_sw128(smem_u32(ds_s) + (uint32_t)t * 2 * kTileBytes, kTileBytes, 1024);
          if (elect_one()) {
            mma_ss_imm<false>(tmem + kColDQ, ad, kd, idesc_q);
#pragma unroll
            for (int ks = 1; ks < kTileRows / 16; ++ks)
              if (ks < ksteps) mma_ss_imm<true>(tmem + kColDQ, ad + (uint64_t)(ks * 128), kd + (uint64_t)(ks * 128), idesc_q);
            mma_commit(smem_u32(&bars->dq_full));
          }
          __syncwarp();
        }
        if (last_jb && has_n) {
          mbar_wait(smem_u32(&bars->acc_full), iter & 1);                          // Q and dO are dead
          load_qdo(n_unit);
        }
      }
    }
  } else {
    // ======================================= pass / drain warps: one key row per thread =======================================
    const int quad = warp;
    const int r = quad * 32 + lane;                       // key row inside the tile == TMEM lane
    const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16);
    const float k2 = scale * 1.4426950408889634f;
    uint32_t iter = 0, dqn = 0;
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      const int b = unit / H, h = unit % H;
      asm volatile("bar.sync 1, 128;" ::: "memory");      // the previous unit's readers of sts / pol_s are done
      for (int i = tid; i < 256; i += 128) {
        float4 st = make_float4(0.f, 0.f, 0.f, 0.f);      // queries past T: P = 0, g = 0
        if (i < T) {
          const float4 raw4 = reinterpret_cast<const float4*>(stats)[(size_t)unit * T + i];
          st = make_float4(-raw4.x, raw4.y, -raw4.w * raw4.y, raw4.z);
        }
        float* e0 = reinterpret_cast<float*>(sts + (i & ~1)) + (i & 1);
        e0[0] = st.x; e0[2] = st.y; e0[4] = st.z; e0[6] = st.w;
        if (kPol) pol_s[i] = i < T ? policy[(size_t)b * T + i] : 0.0f;
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
      for (int jb = 0; jb < kNT; ++jb, ++iter) {
        const int j = jb * kTileRows + r;                 // key token of this thread
        const bool valid = j < T;
        const bool warp_active = jb * kTileRows + quad * 32 < T;
        const float pj = kPol ? pol_s[j & 255] : 1.0f;
        const float gc = (g_cls != nullptr && valid) ? g_cls[(size_t)unit * T + j] : 0.0f;
        float dpol0 = 0.f, dpol1 = 0.f;
        mbar_wait(smem_u32(&bars->sdp_full), iter & 1);
        tc_fence_after();
        if (warp_active) {
          uint32_t nsv[16], ndv[16];
          tmem_ld16_nowait(lane_addr + kColS, nsv);
          tmem_ld16_nowait(lane_addr + kColDP, ndv);
          for (int c = 0; c < nchunks; ++c) {
            uint32_t sv[16], dv[16];
            tmem_ld_wait();
#pragma unroll
            for (int q = 0; q < 16; ++q) { sv[q] = nsv[q]; dv[q] = ndv[q]; }
            if (c + 1 < nchunks) {           // the next chunk's S^T / dP^T columns travel while this one is processed
              tmem_ld16_nowait(lane_addr + kColS + (uint32_t)((c + 1) * 16), nsv);
              tmem_ld16_nowait(lane_addr + kColDP + (uint32_t)((c + 1) * 16), ndv);
            }
            if (c == 0) dv[0] = __float_as_uint(__uint_as_float(dv[0]) + gc);       // d loss / d P[0, j] (CLS-row output)
            // the diagonal (mask 1 whatever the policy) lies in one chunk per thread: warp-uniform split of the two forms
            const bool diag_chunk = kPol && (c * 16 < jb * kTileRows + quad * 32 + 32) && (c * 16 + 16 > jb * kTileRows + quad * 32);
            float pv[16], dsv[16];
            if (diag_chunk) {
#pragma unroll
              for (int q = 0; q < 16; ++q) {
                const int i = c * 16 + q;
                const float* st = reinterpret_cast<const float*>(sts + (i & ~1)) + (i & 1);     // (-m', 1/den, -delta/den, c/den) at +0,2,4,6
                const float et = ex2_approx(fmaf(__uint_as_float(sv[q]), k2, st[0]));
                const float g = fmaf(__uint_as_float(dv[q]), st[2], st[4]);
                const float e = (i == j) ? et : et * pj;
                pv[q] = fmaf(e, st[2], st[6]);
                dsv[q] = g * e;
                const float u = (i == j) ? 0.f : g * et;
                if (q & 1) dpol1 += u; else dpol0 += u;
              }
            } else {
              // two queries per step on the packed fp32x2 pipe (FFMA2 / FMUL2 / FADD2): 7 arithmetic issue slots per pair
              const uint64_t k22 = f2_bcast(k2), pj2 = f2_bcast(pj);
              uint64_t dacc = f2_pack(dpol0, dpol1);
#pragma unroll
              for (int q = 0; q < 16; q += 2) {
                const float4 sa = sts[c * 16 + q], sb = sts[c * 16 + q + 1];
                const uint64_t a2 = f2_pack(sa.z, sa.w);
                float x0, x1;
                f2_unpack(f2_fma(f2_pack(__uint_as_float(sv[q]), __uint_as_float(sv[q + 1])), k22, f2_pack(sa.x, sa.y)), x0, x1);
                const uint64_t et2 = f2_pack(ex2_approx(x0), ex2_approx(x1));
                const uint64_t g2 = f2_fma(f2_pack(__uint_as_float(dv[q]), __uint_as_float(dv[q + 1])), a2, f2_pack(sb.x, sb.y));
                const uint64_t u2 = f2_mul(g2, et2);
                const uint64_t e2 = kPol ? f2_mul(et2, pj2) : et2;
                f2_unpack(f2_fma(e2, a2, f2_pack(sb.z, sb.w)), pv[q], pv[q + 1]);
                f2_unpack(kPol ? f2_mul(u2, pj2) : u2, dsv[q], dsv[q + 1]);
                if (kPol) dacc = f2_add(dacc, u2);
              }
              if (kPol) f2_unpack(dacc, dpol0, dpol1);
            }
            uint32_t pp[8], dd[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              // key rows past T hold whatever the zero-filled K / V rows produce: force exact zeros (0 * NaN would reach dQ)
              pp[q] = valid ? pack_bf16x2(pv[2 * q], pv[2 * q + 1]) : 0u;
              dd[q] = valid ? pack_bf16x2(dsv[2 * q], dsv[2 * q + 1]) : 0u;
            }
            tmem_st8(lane_addr + kColS + (uint32_t)(c * 8), pp);     // overlays S^T / dP^T columns already consumed
            tmem_st8(lane_addr + kColDP + (uint32_t)(c * 8), dd);
            unsigned char* blk = ds_s + (size_t)(c >> 2) * kTileBytes;
            const int cc = (c & 3) * 2;
            *reinterpret_cast<uint4*>(blk + sw128_off(r, cc)) = make_uint4(dd[0], dd[1], dd[2], dd[3]);
            *reinterpret_cast<uint4*>(blk + sw128_off(r, cc + 1)) = make_uint4(dd[4], dd[5], dd[6], dd[7]);
          }
          if (kPol && valid) atomicAdd(&gpolicy[(size_t)b * T + j], dpol0 + dpol1);
        }
        tmem_st_wait();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");               // dS tile -> visible to the MMA
        tc_fence_before();
        mbar_arrive(smem_u32(&bars->pds_full));

        // ---- dV_jb, dK_jb: this thread's key row, 64 columns each ----------------------------------------------------
        mbar_wait(smem_u32(&bars->acc_full), iter & 1);
        tc_fence_after();
        if (warp_active) {
#pragma unroll
          for (int which = 0; which < 2; ++which) {       // 0: dK (scaled), 1: dV
            const uint32_t col = which == 0 ? kColDK : kColDV;
            const float f = which == 0 ? scale : 1.0f;
            uint4* dst = reinterpret_cast<uint4*>(dqkv + ((size_t)b * T + (valid ? j : 0)) * (size_t)(3 * H * kTcHD) +
                                                  (size_t)((1 + which) * H + h) * kTcHD);
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {
              uint32_t v[16];
              tmem_ld16_nowait(lane_addr + col + (uint32_t)(ch * 16), v);
              tmem_ld_wait();
              uint32_t w[8];
#pragma unroll
              for (int q = 0; q < 8; ++q) w[q] = pack_bf16x2(__uint_as_float(v[2 * q]) * f, __uint_as_float(v[2 * q + 1]) * f);
              if (valid) {
                dst[ch * 2] = make_uint4(w[0], w[1], w[2], w[3]);
                dst[ch * 2 + 1] = make_uint4(w[4], w[5], w[6], w[7]);
              }
            }
          }
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&bars->acc_free));

        // ---- dQ_t: this thread's QUERY row i = 128 t + r -------------------------------------------------------------
#pragma unroll
        for (int t = 0; t < kNT; ++t, ++dqn) {
          const int i = t * kTileRows + r;
          const bool q_active = t * kTileRows + quad * 32 < T;
          mbar_wait(smem_u32(&bars->dq_full), dqn & 1);
          tc_fence_after();
          if (q_active) {
            float4* st4 = reinterpret_cast<float4*>(stash) + (size_t)i * 16;       // 16 x 16 B per row, chunk index xor (row & 15)
            uint4* dst = reinterpret_cast<uint4*>(dqkv + ((size_t)b * T + (i < T ? i : 0)) * (size_t)(3 * H * kTcHD) + (size_t)h * kTcHD);
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {
              uint32_t v[16];
              tmem_ld16_nowait(lane_addr + kColDQ + (uint32_t)(ch * 16), v);
              tmem_ld_wait();
              if (kNT == 2 && jb == 0) {
                if (i < T) {
#pragma unroll
                  for (int q = 0; q < 4; ++q)
                    st4[(ch * 4 + q) ^ (i & 15)] = make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]),
                                                               __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
                }
              } else {
                float o[16];
#pragma unroll
                for (int q = 0; q < 16; ++q) o[q] = __uint_as_float(v[q]);
                if (kNT == 2 && i < T) {
#pragma unroll
                  for (int q = 0; q < 4; ++q) {
                    const float4 p = st4[(ch * 4 + q) ^ (i & 15)];
                    o[4 * q] += p.x; o[4 * q + 1] += p.y; o[4 * q + 2] += p.z; o[4 * q + 3] += p.w;
                  }
                }
                uint32_t w[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) w[q] = pack_bf16x2(o[2 * q] * scale, o[2 * q + 1] * scale);
                if (i < T) {
                  dst[ch * 2] = make_uint4(w[0], w[1], w[2], w[3]);
                  dst[ch * 2 + 1] = make_uint4(w[4], w[5], w[6], w[7]);
                }
              }
            }
          }
          tc_fence_before();
          mbar_arrive(smem_u32(&bars->dq_free));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512) : "memory");
  }
}

static size_t bwd_smem_bytes(int knt, int Tp) {
  return 1024 + (size_t)2 * Tp * 128 + (size_t)(3 + 2 * knt) * kTileBytes + (knt == 2 ? (size_t)Tp * kTcHD * 4 : 0) + 256 * 16 +
         256 * 4 + sizeof(BwdBars);
}

// the delta pre-pass of both training backwards (d2s_attn_policy_bwd, d2s_attn_long_bwd): stats[..][3] = gout_i . out_i (+ g_cls . P_0)
int launch_attn_bwd_prep(const void* out, const void* gout, const float* cls_row, const float* g_cls, int B, int T, int H,
                         float* stats, cudaStream_t stream) {
  const long long rows = (long long)B * T * H;
  attn_bwd_prep_kernel<<<(unsigned)((rows + 31) / 32), 256, 0, stream>>>((const __nv_bfloat16*)out, (const __nv_bfloat16*)gout,
                                                                          cls_row, g_cls, rows, T, H, stats);
  count_launch();
  return check_launch("attn_bwd_prep");
}

template <int kNT, bool kPol>
static int launch_bwd(const CUtensorMap* maps, const float* policy, const float* stats, const float* g_cls, int units, int T, int H,
                      int Tp, float scale, void* dqkv, float* gpolicy, cudaStream_t stream) {
  auto kern = attn_tc_bwd_kernel<kNT, kPol>;
  const size_t smem = bwd_smem_bytes(kNT, Tp);
  static SmemOptIn opt;   // one per instantiation: opt in to the size the largest T of this variant needs
  cudaError_t e = opt_in_smem(opt, kern, (int)bwd_smem_bytes(kNT, kNT == 1 ? kTileRows : kBwdMaxT));
  D2S_REQUIRE(e == cudaSuccess, D2S_ERR_CUDA, "attn_policy_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  const int grid = units < kNumSMs ? units : kNumSMs;
  kern<<<grid, kBwdThreads, smem, stream>>>(maps[0], maps[1], maps[2], maps[3], policy, stats, g_cls, units, T, H, Tp, scale,
                                            (__nv_bfloat16*)dqkv, gpolicy);
  count_launch();
  return check_launch("d2s_attn_policy_bwd(tcgen05)");
}

}  // namespace d2s

using namespace d2s;

extern "C" int d2s_attn_policy_bwd(const void* qkv, const float* policy, const void* out, const void* gout, const float* cls_row,
                                   const float* g_cls, float* stats, int B, int T, int H, int hd, float scale, void* dqkv,
                                   float* gpolicy, d2s_stream_t stream_) {
  D2S_REQUIRE(qkv && out && gout && stats && dqkv, D2S_ERR_ARG, "attn_policy_bwd: null pointer");
  D2S_REQUIRE((policy == nullptr) == (gpolicy == nullptr), D2S_ERR_ARG, "attn_policy_bwd: policy and gpolicy go together");
  D2S_REQUIRE(g_cls == nullptr || cls_row != nullptr, D2S_ERR_ARG, "attn_policy_bwd: g_cls needs the forward's cls_row");
  D2S_REQUIRE(B >= 0 && T >= 1 && H >= 1, D2S_ERR_ARG, "attn_policy_bwd: bad shape B=%d T=%d H=%d", B, T, H);
  D2S_REQUIRE(hd == kTcHD, D2S_ERR_ARG, "attn_policy_bwd: head dim %d unsupported (64 only)", hd);
  D2S_REQUIRE(T <= kBwdMaxT, D2S_ERR_ARG, "attn_policy_bwd: T=%d exceeds %d", T, kBwdMaxT);
  D2S_REQUIRE((long long)B * H <= (1LL << 30), D2S_ERR_ARG, "attn_policy_bwd: B*H=%lld too large", (long long)B * H);
  D2S_REQUIRE(scale > 0.0f, D2S_ERR_ARG, "attn_policy_bwd: scale must be positive (got %g)", (double)scale);
  D2S_REQUIRE(aligned16(qkv) && aligned16(out) && aligned16(gout) && aligned16(stats) && aligned16(dqkv), D2S_ERR_ALIGN,
              "attn_policy_bwd: qkv/out/gout/stats/dqkv must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  cudaStream_t stream = (cudaStream_t)stream_;
  GgEncodeFn enc = gg_encode_fn();
  D2S_REQUIRE(enc != nullptr, D2S_ERR_CUDA, "attn_policy_bwd: cuTensorMapEncodeTiled is unavailable from the driver");
  const int Tp = ceil_div(T, 16) * 16;
  const int rows_a = Tp < kTileRows ? Tp : kTileRows;
  const int rows_b = Tp > kTileRows ? Tp - kTileRows : rows_a;
  // maps 0/1: packed qkv (3*H*64 columns, T tokens, B images), boxes of rows_a / rows_b rows; maps 2/3: the same over dO (H*64)
  CUtensorMap maps[4];
  for (int m = 0; m < 4; ++m) {
    const int cols = (m < 2 ? 3 : 1) * H * kTcHD;
    const cuuint64_t gdim[3] = {(cuuint64_t)cols, (cuuint64_t)T, (cuuint64_t)B};
    const cuuint64_t gstride[2] = {(cuuint64_t)cols * 2, (cuuint64_t)T * cols * 2};
    const cuuint32_t estr[3] = {1, 1, 1};
    const cuuint32_t box[3] = {(cuuint32_t)kTcHD, (cuuint32_t)((m & 1) == 0 ? rows_a : rows_b), 1};
    CUresult cr = enc(&maps[m], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(m < 2 ? qkv : gout), gdim, gstride, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    D2S_REQUIRE(cr == CUDA_SUCCESS, D2S_ERR_CUDA, "attn_policy_bwd: cuTensorMapEncodeTiled failed (%d)", (int)cr);
  }
  const int rc = launch_attn_bwd_prep(out, gout, cls_row, g_cls, B, T, H, stats, stream);
  if (rc != D2S_OK) return rc;
  const int units = B * H;
  if (T <= kTileRows)
    return policy ? launch_bwd<1, true>(maps, policy, stats, g_cls, units, T, H, Tp, scale, dqkv, gpolicy, stream)
                  : launch_bwd<1, false>(maps, policy, stats, g_cls, units, T, H, Tp, scale, dqkv, gpolicy, stream);
  return policy ? launch_bwd<2, true>(maps, policy, stats, g_cls, units, T, H, Tp, scale, dqkv, gpolicy, stream)
                : launch_bwd<2, false>(maps, policy, stats, g_cls, units, T, H, Tp, scale, dqkv, gpolicy, stream);
}
