// Attention backward beyond 208 tokens (d2s_attn_long_bwd): the backward of d2s_attn_long_fwd_stats / d2s_attn_policy_fwd for
// 1 <= T <= 2048, bf16 in, fp32 accumulate, hd = 64, key-blocked on tcgen05 / TMEM.  Semantics are exactly those of
// d2s_attn_policy_bwd (header comment of d2s_attn_bwd.cu): scores and probabilities are recomputed from qkv and the forward's
// row statistics, g = (dP - delta) / den, dS = g e~ m, d p_j = sum_h sum_{i != j} g_ij e~_ij, delta includes g_cls . P_0, and
// the O(eps) gradient through the subtracted row maximum is dropped.  No T x T tensor touches global memory.
//
//   unit      = (image, head); one persistent CTA per SM walks its units, and per unit
//   for each 128-key tile jt  (K_jt, V_jt loaded once):
//     for each 128-query block qb  (Q_qb, dO_qb through a two-stage TMA ring):
//       S^T  = K_jt Q_qb^T        dP^T = V_jt dO_qb^T           (SS, TMEM lanes = keys, columns = queries)
//       pass: P^T, dS^T packed bf16 over the consumed columns; dS^T also to a SWIZZLE_128B shared tile; d policy per thread
//       dV  += P^T dO_qb          dK  += dS^T Q_qb              (TS, accumulated over query blocks in TMEM)
//       dQ_qb = dS K_jt                                         (SS, A = the MN-major dS^T tile)
//       dQ_qb drained by its query-row thread: read-add-write of an fp32 (B,H,T,64) workspace, in key-tile order (deterministic);
//       the last key tile writes scale dQ as bf16 into dqkv
//     dK (scaled), dV of the tile to dqkv; one atomicAdd of d policy per key
//
// TMEM (512 columns, one CTA per SM): S^T / P^T [0,128), dP^T / dS^T [128,256), dV [256,320), dK [320,384), dQ [384,448).
// Warps 0-3: pass / drains (one key row per thread for the pass and dK / dV, one query row per thread for dQ; TMEM lane
// quadrant = warp); warp 4: MMA issue; warp 5: TMA producer.  The steps of one (key tile, query block) run one after another
// (S^T and dP^T of the next block overwrite this block's P^T / dS^T, so they wait for its dK / dV / dQ MMAs); only the TMA
// loads run ahead.  Nothing in shared memory is T-sized, so 2048 is a choice matching the forward, not a capacity limit.
#include "d2s_tc.cuh"

namespace d2s {
namespace {

constexpr int kLbMaxT = 2048;
constexpr int kLbThreads = 6 * 32;            // 4 pass / drain warps, MMA warp, TMA warp
constexpr int kLbMmaWarp = 4, kLbTmaWarp = 5;
constexpr uint32_t kLbS = 0, kLbDP = 128, kLbDV = 256, kLbDK = 320, kLbDQ = 384;   // TMEM columns

struct LongBwdBars {
  uint64_t qdo_full[2], qdo_empty[2], kv_full, kv_empty, sdp_full, pds_full, dq_full, dq_free, acc_full, acc_free;
  uint32_t tmem_base;
  uint32_t pad;
};

// shared memory after the 1024-byte alignment pad: Q ring, dO ring, K, V, dS^T (two 64-query blocks), statistics, barriers
constexpr size_t kLbSmem = 1024 + 8 * (size_t)kTileBytes + kTileRows * 16 + sizeof(LongBwdBars);

struct LbShape {
  int T, H, nt;      // tokens, heads, 128-row tiles per (image, head) -- key tiles and query blocks alike
};

// chunks of 16 rows of tile t that hold valid tokens (1..8)
__device__ __forceinline__ int tile_chunks(int T, int t) { return min(8, (T - t * kTileRows + 15) >> 4); }

template <bool kPol>
__global__ void __launch_bounds__(kLbThreads, 1)
attn_long_bwd_kernel(const __grid_constant__ CUtensorMap map_qkv, const __grid_constant__ CUtensorMap map_go,
                     const float* __restrict__ policy, const float* __restrict__ stats, const float* __restrict__ g_cls,
                     int num_units, LbShape shp, float scale, __nv_bfloat16* __restrict__ dqkv, float* __restrict__ gpolicy,
                     float* __restrict__ ws) {
  extern __shared__ unsigned char smem_dyn[];
  const uint32_t raw = smem_u32(smem_dyn);
  unsigned char* tiles = smem_dyn + ((1024u - (raw & 1023u)) & 1023u);   // SWIZZLE_128B atoms are address based
  unsigned char* q_s = tiles;                       // 2 stages x 128 query rows x 128 B
  unsigned char* do_s = q_s + 2 * kTileBytes;       // 2 stages
  unsigned char* k_s = do_s + 2 * kTileBytes;
  unsigned char* v_s = k_s + kTileBytes;
  unsigned char* ds_s = v_s + kTileBytes;           // [64-query block][128 key rows][128 B]
  // per-query statistics of the current block, two queries per entry for the packed fp32x2 arithmetic of the pass (as in
  // d2s_attn_bwd.cu): sts[2 p] = (-m'_i, -m'_i+1, 1/den_i, 1/den_i+1), sts[2 p + 1] = (-delta_i/den_i, .., c_i/den_i, ..), i = 2 p
  float4* sts = reinterpret_cast<float4*>(ds_s + 2 * kTileBytes);
  LongBwdBars* bars = reinterpret_cast<LongBwdBars*>(sts + kTileRows);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int T = shp.T, H = shp.H, nt = shp.nt;
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_u32(&bars->qdo_full[s]), 1);
      mbar_init(smem_u32(&bars->qdo_empty[s]), 1);
    }
    mbar_init(smem_u32(&bars->kv_full), 1);
    mbar_init(smem_u32(&bars->kv_empty), 1);
    mbar_init(smem_u32(&bars->sdp_full), 1);
    mbar_init(smem_u32(&bars->pds_full), 128);
    mbar_init(smem_u32(&bars->dq_full), 1);
    mbar_init(smem_u32(&bars->dq_free), 128);
    mbar_init(smem_u32(&bars->acc_full), 1);
    mbar_init(smem_u32(&bars->acc_free), 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kLbMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)), "n"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;

  const int w = warp_uniform(warp);
  if (w == kLbTmaWarp) {
    // ================= TMA producer: K_jt / V_jt once per key tile, Q_qb / dO_qb of every query block through the ring =======
    uint32_t it = 0, kvn = 0;
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      const int b = unit / H, h = unit - (unit / H) * H;
      for (int jt = 0; jt < nt; ++jt, ++kvn) {
        if (kvn > 0) mbar_wait(smem_u32(&bars->kv_empty), (kvn - 1) & 1);
        if (elect_one()) {
          mbar_expect_tx(smem_u32(&bars->kv_full), 2 * kTileBytes);
          tma_load_3d(smem_u32(k_s), &map_qkv, (H + h) * kTcHD, jt * kTileRows, b, smem_u32(&bars->kv_full));
          tma_load_3d(smem_u32(v_s), &map_qkv, (2 * H + h) * kTcHD, jt * kTileRows, b, smem_u32(&bars->kv_full));
        }
        __syncwarp();
        for (int qb = 0; qb < nt; ++qb, ++it) {
          const uint32_t st = it & 1;
          if (it >= 2) mbar_wait(smem_u32(&bars->qdo_empty[st]), ((it >> 1) - 1) & 1);
          if (elect_one()) {
            mbar_expect_tx(smem_u32(&bars->qdo_full[st]), 2 * kTileBytes);
            tma_load_3d(smem_u32(q_s + st * kTileBytes), &map_qkv, h * kTcHD, qb * kTileRows, b, smem_u32(&bars->qdo_full[st]));
            tma_load_3d(smem_u32(do_s + st * kTileBytes), &map_go, h * kTcHD, qb * kTileRows, b, smem_u32(&bars->qdo_full[st]));
          }
          __syncwarp();
        }
      }
    }
  } else if (w == kLbMmaWarp) {
    // ================= MMA issue: warp-uniform loop, one elected lane per instruction =================
    const uint32_t idesc_s = make_idesc(kTileRows, kTileRows, 0);   // S^T, dP^T: M = keys, N = queries
    const uint32_t idesc_kv = make_idesc(kTileRows, kTcHD, 1);      // dV, dK: A from TMEM, B MN-major
    const uint32_t idesc_q = make_idesc(kTileRows, kTcHD, 1, 1);    // dQ: A and B MN-major
    const uint64_t kd = make_desc_sw128(smem_u32(k_s), 16, 1024), vd = make_desc_sw128(smem_u32(v_s), 16, 1024);
    // A = dS, M = 128 queries: two 64-query blocks 16 KB apart (LBO), 8 key rows per 1024 B (SBO)
    const uint64_t ad = make_desc_sw128(smem_u32(ds_s), kTileBytes, 1024);
    uint32_t it = 0, kvn = 0;
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      for (int jt = 0; jt < nt; ++jt, ++kvn) {
        const int ksteps = tile_chunks(T, jt);                      // key rows of this tile / 16
        for (int qb = 0; qb < nt; ++qb, ++it) {
          const uint32_t st = it & 1;
          const int nch = tile_chunks(T, qb);                       // query columns of this block / 16
          const uint64_t qd = make_desc_sw128(smem_u32(q_s + st * kTileBytes), 16, 1024);
          const uint64_t gd = make_desc_sw128(smem_u32(do_s + st * kTileBytes), 16, 1024);
          mbar_wait(smem_u32(&bars->qdo_full[st]), (it >> 1) & 1);
          if (qb == 0) mbar_wait(smem_u32(&bars->kv_full), kvn & 1);
          if (it > 0) mbar_wait(smem_u32(&bars->dq_full), (it - 1) & 1);   // every MMA of the previous block has completed
          tc_fence_after();
          if (elect_one()) {
            mma_ss_imm<false>(tmem + kLbS, kd, qd, idesc_s);
            mma_ss_imm<true>(tmem + kLbS, kd + 2, qd + 2, idesc_s);
            mma_ss_imm<true>(tmem + kLbS, kd + 4, qd + 4, idesc_s);
            mma_ss_imm<true>(tmem + kLbS, kd + 6, qd + 6, idesc_s);
            mma_ss_imm<false>(tmem + kLbDP, vd, gd, idesc_s);
            mma_ss_imm<true>(tmem + kLbDP, vd + 2, gd + 2, idesc_s);
            mma_ss_imm<true>(tmem + kLbDP, vd + 4, gd + 4, idesc_s);
            mma_ss_imm<true>(tmem + kLbDP, vd + 6, gd + 6, idesc_s);
            mma_commit(smem_u32(&bars->sdp_full));
          }
          __syncwarp();
          mbar_wait(smem_u32(&bars->pds_full), it & 1);             // P^T, dS^T in TMEM; dS in shared memory
          if (qb == 0 && kvn > 0) mbar_wait(smem_u32(&bars->acc_free), (kvn - 1) & 1);   // previous tile's dK / dV drained
          if (it > 0) mbar_wait(smem_u32(&bars->dq_free), (it - 1) & 1);                 // previous block's dQ drained
          tc_fence_after();
          if (elect_one()) {
            if (qb == 0) mma_ts_imm<false>(tmem + kLbDV, tmem + kLbS, gd, idesc_kv);
            else mma_ts_imm<true>(tmem + kLbDV, tmem + kLbS, gd, idesc_kv);
#pragma unroll
            for (int ks = 1; ks < 8; ++ks)
              if (ks < nch) mma_ts_imm<true>(tmem + kLbDV, tmem + kLbS + ks * 8, gd + (uint64_t)(ks * 128), idesc_kv);
            if (qb == 0) mma_ts_imm<false>(tmem + kLbDK, tmem + kLbDP, qd, idesc_kv);
            else mma_ts_imm<true>(tmem + kLbDK, tmem + kLbDP, qd, idesc_kv);
#pragma unroll
            for (int ks = 1; ks < 8; ++ks)
              if (ks < nch) mma_ts_imm<true>(tmem + kLbDK, tmem + kLbDP + ks * 8, qd + (uint64_t)(ks * 128), idesc_kv);
            mma_ss_imm<false>(tmem + kLbDQ, ad, kd, idesc_q);
#pragma unroll
            for (int ks = 1; ks < 8; ++ks)
              if (ks < ksteps) mma_ss_imm<true>(tmem + kLbDQ, ad + (uint64_t)(ks * 128), kd + (uint64_t)(ks * 128), idesc_q);
            mma_commit(smem_u32(&bars->dq_full));
            mma_commit(smem_u32(&bars->qdo_empty[st]));
            if (qb == nt - 1) {
              mma_commit(smem_u32(&bars->acc_full));
              mma_commit(smem_u32(&bars->kv_empty));
            }
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ================= pass / drain warps =================
    const int quad = warp;
    const int r = quad * 32 + lane;                                 // TMEM lane: key row (pass, dK, dV), query row (dQ)
    const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16);
    const float k2 = scale * 1.4426950408889634f;
    uint32_t it = 0, kvn = 0;
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      const int b = unit / H, h = unit - (unit / H) * H;
      for (int jt = 0; jt < nt; ++jt, ++kvn) {
        const int j = jt * kTileRows + r;                           // key token of this thread
        const bool valid = j < T;
        const bool warp_active = jt * kTileRows + quad * 32 < T;
        const float pj = (kPol && valid) ? policy[(size_t)b * T + j] : 1.0f;
        float dpol0 = 0.f, dpol1 = 0.f;
        for (int qb = 0; qb < nt; ++qb, ++it) {
          const int nch = tile_chunks(T, qb);
          asm volatile("bar.sync 1, 128;" ::: "memory");             // the previous block's readers of sts are done
          {
            const int i = qb * kTileRows + r;
            float4 st = make_float4(0.f, 0.f, 0.f, 0.f);            // queries past T: P = 0, g = 0
            if (i < T) {
              const float4 raw4 = reinterpret_cast<const float4*>(stats)[(size_t)unit * T + i];
              st = make_float4(-raw4.x, raw4.y, -raw4.w * raw4.y, raw4.z);
            }
            float* e0 = reinterpret_cast<float*>(sts + (r & ~1)) + (r & 1);
            e0[0] = st.x; e0[2] = st.y; e0[4] = st.z; e0[6] = st.w;
          }
          asm volatile("bar.sync 1, 128;" ::: "memory");
          const float gc = (g_cls != nullptr && qb == 0 && valid) ? g_cls[(size_t)unit * T + j] : 0.0f;
          mbar_wait(smem_u32(&bars->sdp_full), it & 1);
          tc_fence_after();
          if (warp_active) {
            uint32_t nsv[16], ndv[16];
            tmem_ld16_nowait(lane_addr + kLbS, nsv);
            tmem_ld16_nowait(lane_addr + kLbDP, ndv);
            for (int c = 0; c < nch; ++c) {
              uint32_t sv[16], dv[16];
              tmem_ld_wait();
#pragma unroll
              for (int q = 0; q < 16; ++q) { sv[q] = nsv[q]; dv[q] = ndv[q]; }
              if (c + 1 < nch) {             // the next chunk's S^T / dP^T columns travel while this one is processed
                tmem_ld16_nowait(lane_addr + kLbS + (uint32_t)((c + 1) * 16), nsv);
                tmem_ld16_nowait(lane_addr + kLbDP + (uint32_t)((c + 1) * 16), ndv);
              }
              if (c == 0) dv[0] = __float_as_uint(__uint_as_float(dv[0]) + gc);   // d loss / d P[0, j] (query 0: qb == 0 only)
              // the diagonal (mask 1 whatever the policy) lies in one chunk per thread: warp-uniform split of the two forms
              const bool diag_chunk = kPol && qb == jt && (c * 16 < quad * 32 + 32) && (c * 16 + 16 > quad * 32);
              float pv[16], dsv[16];
              if (diag_chunk) {
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                  const int il = c * 16 + q;
                  const float* st = reinterpret_cast<const float*>(sts + (il & ~1)) + (il & 1);   // (-m', 1/den, -delta/den, c/den)
                  const float et = ex2_approx(fmaf(__uint_as_float(sv[q]), k2, st[0]));
                  const float g = fmaf(__uint_as_float(dv[q]), st[2], st[4]);
                  const float e = (il == r) ? et : et * pj;
                  pv[q] = fmaf(e, st[2], st[6]);
                  dsv[q] = g * e;
                  const float u = (il == r) ? 0.f : g * et;
                  if (q & 1) dpol1 += u; else dpol0 += u;
                }
              } else {
                // two queries per step on the packed fp32x2 pipe (FFMA2 / FMUL2 / FADD2)
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
              tmem_st8(lane_addr + kLbS + (uint32_t)(c * 8), pp);    // overlays S^T / dP^T columns already consumed
              tmem_st8(lane_addr + kLbDP + (uint32_t)(c * 8), dd);
              unsigned char* blk = ds_s + (size_t)(c >> 2) * kTileBytes;
              const int cc = (c & 3) * 2;
              *reinterpret_cast<uint4*>(blk + sw128_off(r, cc)) = make_uint4(dd[0], dd[1], dd[2], dd[3]);
              *reinterpret_cast<uint4*>(blk + sw128_off(r, cc + 1)) = make_uint4(dd[4], dd[5], dd[6], dd[7]);
            }
          }
          tmem_st_wait();
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // dS tile -> visible to the MMA
          tc_fence_before();
          mbar_arrive(smem_u32(&bars->pds_full));

          // ---- dQ_qb: this thread's QUERY row, accumulated over key tiles in the workspace in key-tile order -------------
          mbar_wait(smem_u32(&bars->dq_full), it & 1);
          tc_fence_after();
          {
            const int i = qb * kTileRows + r;
            if (qb * kTileRows + quad * 32 < T) {
              float4* wrow = reinterpret_cast<float4*>(ws + ((size_t)unit * T + (i < T ? i : 0)) * kTcHD);
              uint4* dst = reinterpret_cast<uint4*>(dqkv + ((size_t)b * T + (i < T ? i : 0)) * (size_t)(3 * H * kTcHD) +
                                                    (size_t)h * kTcHD);
#pragma unroll
              for (int ch = 0; ch < 4; ++ch) {
                uint32_t v[16];
                tmem_ld16_nowait(lane_addr + kLbDQ + (uint32_t)(ch * 16), v);
                tmem_ld_wait();
                float o[16];
#pragma unroll
                for (int q = 0; q < 16; ++q) o[q] = __uint_as_float(v[q]);
                if (i < T) {
                  if (jt > 0) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                      const float4 p = wrow[ch * 4 + q];
                      o[4 * q] = p.x + o[4 * q]; o[4 * q + 1] = p.y + o[4 * q + 1];
                      o[4 * q + 2] = p.z + o[4 * q + 2]; o[4 * q + 3] = p.w + o[4 * q + 3];
                    }
                  }
                  if (jt + 1 < nt) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) wrow[ch * 4 + q] = make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
                  } else {
                    uint32_t wq[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) wq[q] = pack_bf16x2(o[2 * q] * scale, o[2 * q + 1] * scale);
                    dst[ch * 2] = make_uint4(wq[0], wq[1], wq[2], wq[3]);
                    dst[ch * 2 + 1] = make_uint4(wq[4], wq[5], wq[6], wq[7]);
                  }
                }
              }
            }
          }
          tc_fence_before();
          mbar_arrive(smem_u32(&bars->dq_free));
        }

        // ---- end of the key tile: d policy, then dK (scaled) and dV of this thread's key row ---------------------------
        if (kPol && valid) atomicAdd(&gpolicy[(size_t)b * T + j], dpol0 + dpol1);
        mbar_wait(smem_u32(&bars->acc_full), kvn & 1);
        tc_fence_after();
        if (warp_active) {
#pragma unroll
          for (int which = 0; which < 2; ++which) {         // 0: dK (scaled), 1: dV
            const uint32_t col = which == 0 ? kLbDK : kLbDV;
            const float f = which == 0 ? scale : 1.0f;
            uint4* dst = reinterpret_cast<uint4*>(dqkv + ((size_t)b * T + (valid ? j : 0)) * (size_t)(3 * H * kTcHD) +
                                                  (size_t)((1 + which) * H + h) * kTcHD);
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {
              uint32_t v[16];
              tmem_ld16_nowait(lane_addr + col + (uint32_t)(ch * 16), v);
              tmem_ld_wait();
              uint32_t wv[8];
#pragma unroll
              for (int q = 0; q < 8; ++q) wv[q] = pack_bf16x2(__uint_as_float(v[2 * q]) * f, __uint_as_float(v[2 * q + 1]) * f);
              if (valid) {
                dst[ch * 2] = make_uint4(wv[0], wv[1], wv[2], wv[3]);
                dst[ch * 2 + 1] = make_uint4(wv[4], wv[5], wv[6], wv[7]);
              }
            }
          }
        }
        tc_fence_before();
        mbar_arrive(smem_u32(&bars->acc_free));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kLbMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512) : "memory");
  }
}

template <bool kPol>
int launch_long_bwd(const CUtensorMap* maps, const float* policy, const float* stats, const float* g_cls, int units, LbShape shp,
                    float scale, void* dqkv, float* gpolicy, float* ws, cudaStream_t stream) {
  auto kern = attn_long_bwd_kernel<kPol>;
  static SmemOptIn opt;   // one per instantiation
  cudaError_t e = opt_in_smem(opt, kern, (int)kLbSmem);
  D2S_REQUIRE(e == cudaSuccess, D2S_ERR_CUDA, "attn_long_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  const int grid = units < kNumSMs ? units : kNumSMs;
  kern<<<grid, kLbThreads, kLbSmem, stream>>>(maps[0], maps[1], policy, stats, g_cls, units, shp, scale, (__nv_bfloat16*)dqkv,
                                              gpolicy, ws);
  count_launch();
  return check_launch("d2s_attn_long_bwd(tcgen05)");
}

}  // namespace
}  // namespace d2s

using namespace d2s;

extern "C" int d2s_attn_long_bwd(const void* qkv, const float* policy, const void* out, const void* gout, const float* cls_row,
                                 const float* g_cls, float* stats, int B, int T, int H, int hd, float scale, void* dqkv,
                                 float* gpolicy, float* workspace, d2s_stream_t stream_) {
  D2S_REQUIRE(qkv && out && gout && stats && dqkv && workspace, D2S_ERR_ARG, "attn_long_bwd: null pointer");
  D2S_REQUIRE((policy == nullptr) == (gpolicy == nullptr), D2S_ERR_ARG, "attn_long_bwd: policy and gpolicy go together");
  D2S_REQUIRE(g_cls == nullptr || cls_row != nullptr, D2S_ERR_ARG, "attn_long_bwd: g_cls needs the forward's cls_row");
  D2S_REQUIRE(hd == kTcHD, D2S_ERR_ARG, "attn_long_bwd: head dim %d unsupported (64 only)", hd);
  D2S_REQUIRE(B >= 0 && H >= 1 && T >= 1 && T <= kLbMaxT, D2S_ERR_ARG, "attn_long_bwd: bad shape B=%d T=%d H=%d (1 <= T <= %d)", B, T,
              H, kLbMaxT);
  D2S_REQUIRE((long long)B * H <= (1LL << 30), D2S_ERR_ARG, "attn_long_bwd: B*H=%lld too large", (long long)B * H);
  D2S_REQUIRE(scale > 0.0f, D2S_ERR_ARG, "attn_long_bwd: scale must be positive (got %g)", (double)scale);
  D2S_REQUIRE(aligned16(qkv) && aligned16(out) && aligned16(gout) && aligned16(stats) && aligned16(dqkv) && aligned16(workspace),
              D2S_ERR_ALIGN, "attn_long_bwd: qkv/out/gout/stats/dqkv/workspace must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  GgEncodeFn enc = gg_encode_fn();
  D2S_REQUIRE(enc != nullptr, D2S_ERR_CUDA, "attn_long_bwd: cuTensorMapEncodeTiled is unavailable from the driver");
  // map 0: packed qkv (3*H*64 columns, T tokens, B images); map 1: gout (H*64 columns); box 64 x 128 rows, rows past T zero-filled
  CUtensorMap maps[2];
  for (int m = 0; m < 2; ++m) {
    const int cols = (m == 0 ? 3 : 1) * H * kTcHD;
    const cuuint64_t gdim[3] = {(cuuint64_t)cols, (cuuint64_t)T, (cuuint64_t)B};
    const cuuint64_t gstride[2] = {(cuuint64_t)cols * 2, (cuuint64_t)T * cols * 2};
    const cuuint32_t box[3] = {(cuuint32_t)kTcHD, (cuuint32_t)kTileRows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult cr = enc(&maps[m], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(m == 0 ? qkv : gout), gdim, gstride, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    D2S_REQUIRE(cr == CUDA_SUCCESS, D2S_ERR_CUDA, "attn_long_bwd: cuTensorMapEncodeTiled failed (%d)", (int)cr);
  }
  cudaStream_t stream = (cudaStream_t)stream_;
  const int rc = launch_attn_bwd_prep(out, gout, cls_row, g_cls, B, T, H, stats, stream);
  if (rc != D2S_OK) return rc;
  const LbShape shp{T, H, ceil_div(T, kTileRows)};
  const int units = B * H;
  return policy ? launch_long_bwd<true>(maps, policy, stats, g_cls, units, shp, scale, dqkv, gpolicy, workspace, stream)
                : launch_long_bwd<false>(maps, nullptr, stats, g_cls, units, shp, scale, dqkv, gpolicy, workspace, stream);
}
