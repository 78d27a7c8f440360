// Attention forward beyond 256 tokens (d2s_attn_long_fwd): the policy softmax of d2s_attn_policy_fwd for 1 <= T <= 2048, bf16 in,
// fp32 accumulate, hd = 64, key-blocked on tcgen05 / TMEM.  In a translation unit of its own so that the T <= 256 kernels of
// d2s_attn_tc.cu and d2s_attn_varlen.cu compile exactly as before.
//
//   unit      = (image, head, 128-row query tile), numbered so that the query tiles of one (image, head) are adjacent: CTAs
//               resident at the same time re-read that head's K / V from L2
//   per unit  for each 128-column key block j:  S_j = Q K_j^T (TMEM cols [0,128), fp32)
//                                               P_j = exp2(k2 s - m') * mask, packed bf16 (TMEM cols [192,256))
//                                               O  += P_j V_j (TMEM cols [128,192), fp32, A = P from TMEM)
//   out       = (O + eps' colsum(V) / T) / (rowsum + eps')     (dynamic_vit.py:195-214; eps' = eps 2^(k2 max - m'))
//
// Warps 0-3: softmax / epilogue (TMEM lane quadrant = warp); warp 4: tcgen05.mma issue; warp 5: TMA producer.  K and V stream
// through a two-stage ring (box 64 x 128 rows, SWIZZLE_128B, rows past T zero-filled by the TMA unit); nothing T-sized is resident
// except the policy row and the CLS row's un-normalised values (T floats each), so 2048 is a staging limit, not a TMEM one.  Two
// CTAs per SM (256 TMEM columns and ~99 KB of shared memory each): one CTA's MMAs and loads run under the other's exponentials.
//
// Exponent handling is that of the T <= 256 kernel (DESIGN.md section 4 (4)): one whole-binade reference m' from the first 16
// columns of key block 0, the true maximum tracked off the critical path (policy form), NO rescaling of O inside the block loop,
// one test of the finished row sums (beyond 2^100, inf or NaN) after the last block; a failed row is redone from the packed qkv in
// global memory in fp32 over all keys.  A masked key far above every kept one raises m' by whole binades at the end (exact: O, the
// sum and the CLS values are multiplied by the same power of two).
#undef D2S_ATTN_TRACE_BUILD   // the clock64 phase traces instrument the T <= 256 kernels only
#include "d2s_attn_tc.cuh"

namespace d2s {
namespace {

constexpr int kLongMaxT = 2048;
constexpr int kLongStages = 2;                 // K / V ring depth
constexpr int kLongThreads = 6 * 32;           // 4 softmax / epilogue warps, MMA warp, TMA warp
constexpr int kLongMmaWarp = 4, kLongTmaWarp = 5;
constexpr uint32_t kSCol = 0, kOCol = 128, kPCol = 192;   // TMEM columns: S block, O accumulator, packed P block
constexpr int kLongTmemCols = 256;

struct alignas(16) LongBars {   // 16-byte multiple: the policy row behind it is read as float4
  uint64_t q_full, q_empty;
  uint64_t k_full[kLongStages], k_empty[kLongStages], v_full[kLongStages], v_empty[kLongStages];
  uint64_t s_full, p_full, pv_done, o_free;
  uint32_t tmem_base;
};

// shared memory after the 1024-byte alignment pad: Q tile, K ring, V ring, barriers, policy row, CLS row, colsum(V) partials
constexpr size_t kLongTileRegion = (size_t)(1 + 2 * kLongStages) * kTileBytes;
constexpr size_t kLongSmem = 1024 + kLongTileRegion + sizeof(LongBars) + (2 * kLongMaxT + 3 * kTcHD) * sizeof(float);

struct LongShape {
  int T, H, nqt;     // padded length, heads, query tiles per (image, head)
  __device__ __forceinline__ void decode(int unit, int& b, int& h, int& qt) const {
    const int bh = unit / nqt;
    qt = unit - bh * nqt;
    b = bh / H;
    h = bh - b * H;
  }
};

// valid tokens of image b (T in the dense form)
template <bool kVar>
__device__ __forceinline__ int long_len(const int* __restrict__ lens, int b, int T) { return kVar ? var_len(lens, b, T) : T; }
// 16-key chunks of key block jb holding valid keys (1..8)
__device__ __forceinline__ int block_chunks(int Tv, int jb) { return min(8, (Tv - jb * 128 + 15) >> 4); }

// kPol: policy given (eps terms, masked exponentials, colsum(V)).  kVar: variable-length form (lens, no policy).
template <bool kPol, bool kVar>
__global__ void __launch_bounds__(kLongThreads, 2)
attn_long_fwd_kernel(const __grid_constant__ CUtensorMap map, const float* __restrict__ policy, const int* __restrict__ lens,
                     int num_units, LongShape shp, float scale, float eps, __nv_bfloat16* __restrict__ out,
                     float* __restrict__ cls_row, const __nv_bfloat16* __restrict__ qkv) {
  static_assert(!(kVar && kPol), "the variable-length form takes no policy");
  extern __shared__ unsigned char smem_dyn[];
  const uint32_t raw = smem_u32(smem_dyn);
  unsigned char* tiles = smem_dyn + ((1024u - (raw & 1023u)) & 1023u);   // SWIZZLE_128B atoms are address based
  unsigned char* q_s = tiles;
  unsigned char* k_s = q_s + kTileBytes;                        // kLongStages x 128 rows x 128 B
  unsigned char* v_s = k_s + kLongStages * kTileBytes;          // kLongStages x 128 rows x 128 B
  LongBars* bars = reinterpret_cast<LongBars*>(v_s + kLongStages * kTileBytes);
  float* pol_s = reinterpret_cast<float*>(bars + 1);            // kLongMaxT: policy row, zeros past T
  float* cls_s = pol_s + kLongMaxT;                             // kLongMaxT: un-normalised values of query row 0
  float* vpart_s = cls_s + kLongMaxT;                           // 2 x 64 partial column sums of V
  float* vsum_s = vpart_s + 2 * kTcHD;                          // 64

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int T = shp.T, H = shp.H;

  if (tid == 0) {
    mbar_init(smem_u32(&bars->q_full), 1);
    mbar_init(smem_u32(&bars->q_empty), 1);
    for (int s = 0; s < kLongStages; ++s) {
      mbar_init(smem_u32(&bars->k_full[s]), 1);
      mbar_init(smem_u32(&bars->k_empty[s]), 1);
      mbar_init(smem_u32(&bars->v_full[s]), 1);
      mbar_init(smem_u32(&bars->v_empty[s]), kPol ? 1 + 128 : 1);   // policy form: the softmax warps also read V (colsum)
    }
    mbar_init(smem_u32(&bars->s_full), 1);
    mbar_init(smem_u32(&bars->p_full), 128);
    mbar_init(smem_u32(&bars->pv_done), 1);
    mbar_init(smem_u32(&bars->o_free), 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kLongMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)),
                 "n"(kLongTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;

  const int w = warp_uniform(warp);
  if (w == kLongTmaWarp) {
    // ================= TMA producer: Q once per unit, then K_j / V_j of every key block through the ring =================
    uint32_t g = 0, qn = 0;
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      int b, h, qt;
      shp.decode(unit, b, h, qt);
      const int Tv = long_len<kVar>(lens, b, T);
      if (qt * kTileRows >= Tv) continue;                        // (variable-length form) a tile of pad rows only
      const int nblk = (Tv + kTileRows - 1) / kTileRows;
      if (qn > 0) mbar_wait(smem_u32(&bars->q_empty), (qn - 1) & 1);
      if (elect_one()) {
        mbar_expect_tx(smem_u32(&bars->q_full), kTileBytes);
        tma_load_3d(smem_u32(q_s), &map, h * kTcHD, qt * kTileRows, b, smem_u32(&bars->q_full));
      }
      __syncwarp();
      for (int jb = 0; jb < nblk; ++jb, ++g) {
        const uint32_t st = g % kLongStages, ph = (g / kLongStages) & 1;
        mbar_wait(smem_u32(&bars->k_empty[st]), ph ^ 1);
        if (elect_one()) {
          mbar_expect_tx(smem_u32(&bars->k_full[st]), kTileBytes);
          tma_load_3d(smem_u32(k_s + st * kTileBytes), &map, (H + h) * kTcHD, jb * kTileRows, b, smem_u32(&bars->k_full[st]));
        }
        __syncwarp();
        mbar_wait(smem_u32(&bars->v_empty[st]), ph ^ 1);
        if (elect_one()) {
          mbar_expect_tx(smem_u32(&bars->v_full[st]), kTileBytes);
          tma_load_3d(smem_u32(v_s + st * kTileBytes), &map, (2 * H + h) * kTcHD, jb * kTileRows, b, smem_u32(&bars->v_full[st]));
        }
        __syncwarp();
      }
      ++qn;
    }
  } else if (w == kLongMmaWarp) {
    // ================= MMA issue: warp-uniform loop, one elected lane per instruction (DESIGN.md section 4, "Two lessons") ======
    // Per block j: S_{j+1} is issued as soon as the softmax has consumed S_j (p_full), ahead of PV_j, so that the next block's
    // scores are ready when the softmax warps come back; P_j lives in its own TMEM columns, so S_{j+1} cannot overwrite it.
    const uint32_t idesc_s = make_idesc(kTileRows, kTileRows, 0);
    const uint32_t idesc_o = make_idesc(kTileRows, kTcHD, 1);
    const uint64_t qd = make_desc_sw128(smem_u32(q_s), 16, 1024);
    uint32_t g = 0, qn = 0, un = 0;
    auto issue_s = [&](uint32_t gb) {
      const uint32_t st = gb % kLongStages;
      mbar_wait(smem_u32(&bars->k_full[st]), (gb / kLongStages) & 1);
      tc_fence_after();
      const uint64_t kd = make_desc_sw128(smem_u32(k_s + st * kTileBytes), 16, 1024);
      if (elect_one()) {
        mma_ss_imm<false>(tmem + kSCol, qd, kd, idesc_s);
        mma_ss_imm<true>(tmem + kSCol, qd + 2, kd + 2, idesc_s);
        mma_ss_imm<true>(tmem + kSCol, qd + 4, kd + 4, idesc_s);
        mma_ss_imm<true>(tmem + kSCol, qd + 6, kd + 6, idesc_s);
        mma_commit(smem_u32(&bars->s_full));
        mma_commit(smem_u32(&bars->k_empty[st]));
      }
      __syncwarp();
    };
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      int b, h, qt;
      shp.decode(unit, b, h, qt);
      const int Tv = long_len<kVar>(lens, b, T);
      if (qt * kTileRows >= Tv) continue;
      const int nblk = (Tv + kTileRows - 1) / kTileRows;
      mbar_wait(smem_u32(&bars->q_full), qn & 1);
      issue_s(g);
      if (nblk == 1 && elect_one()) mma_commit(smem_u32(&bars->q_empty));
      __syncwarp();
      for (int jb = 0; jb < nblk; ++jb, ++g) {
        mbar_wait(smem_u32(&bars->p_full), g & 1);             // softmax done with S_j, P_j is in TMEM
        tc_fence_after();
        if (jb + 1 < nblk) {
          issue_s(g + 1);
          if (jb + 2 == nblk && elect_one()) mma_commit(smem_u32(&bars->q_empty));   // Q is dead after the unit's last S-MMA
          __syncwarp();
        }
        if (jb == 0 && un > 0) mbar_wait(smem_u32(&bars->o_free), (un - 1) & 1);  // previous unit's O has been read out
        const uint32_t st = g % kLongStages;
        mbar_wait(smem_u32(&bars->v_full[st]), (g / kLongStages) & 1);
        tc_fence_after();
        const uint64_t vd = make_desc_sw128(smem_u32(v_s + st * kTileBytes), 16, 1024);
        const int ks_b = block_chunks(Tv, jb);                  // K-steps holding valid keys (the last block may be short)
        if (elect_one()) {
          if (jb == 0) mma_ts_imm<false>(tmem + kOCol, tmem + kPCol, vd, idesc_o);
          else mma_ts_imm<true>(tmem + kOCol, tmem + kPCol, vd, idesc_o);
#pragma unroll
          for (int ks = 1; ks < 8; ++ks)
            if (ks < ks_b) mma_ts_imm<true>(tmem + kOCol, tmem + kPCol + (uint32_t)(ks * 8), vd + (uint64_t)(ks * 128), idesc_o);
          mma_commit(smem_u32(&bars->pv_done));
          mma_commit(smem_u32(&bars->v_empty[st]));
        }
        __syncwarp();
      }
      ++qn;
      ++un;
    }
  } else {
    // ================= softmax / epilogue warps: one query row per thread =================
    const int quad = warp;                                      // TMEM lane quadrant
    const int r = quad * 32 + lane;
    const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16);
    const float k2 = scale * 1.4426950408889634f;
    const float c_eps = kPol ? eps / (float)T : 0.0f;
    const float eps_den = kPol ? eps : 0.0f;
    uint32_t g = 0, un = 0;
    for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
      int b, h, qt;
      shp.decode(unit, b, h, qt);
      const int Tv = long_len<kVar>(lens, b, T);
      const int i = qt * kTileRows + r;                         // query token of this thread
      const size_t orow_off = ((size_t)b * T + i) * (size_t)(H * kTcHD) + (size_t)h * kTcHD;
      float* cls_dst = cls_row != nullptr ? cls_row + ((size_t)b * H + h) * T : nullptr;
      if (qt * kTileRows >= Tv) {
        // (variable-length form) a tile of pad rows: zeros, and a zero CLS row for an image without tokens
        if (i < T) {
          uint4* orow = reinterpret_cast<uint4*>(out + orow_off);
#pragma unroll
          for (int q = 0; q < kTcHD / 8; ++q) orow[q] = make_uint4(0u, 0u, 0u, 0u);
        }
        if (cls_dst != nullptr && qt == 0)
          for (int j = r; j < T; j += kTileRows) cls_dst[j] = 0.f;
        continue;
      }
      const int nblk = (Tv + kTileRows - 1) / kTileRows;
      const bool warp_active = qt * kTileRows + quad * 32 < Tv;   // whole warp past the valid rows: no exponentials
      const bool want_cls = cls_dst != nullptr && i == 0;
      if (kPol) {
        asm volatile("bar.sync 1, 128;" ::: "memory");          // the previous unit's readers of pol_s / vsum_s are done
        for (int j = r; j < nblk * kTileRows; j += kTileRows) pol_s[j] = j < T ? policy[(size_t)b * T + j] : 0.f;
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f, mx_true = -INFINITY, mxk = 0.f;
      float vacc = 0.f;                                         // policy form: this thread's share of colsum(V)
      for (int jb = 0; jb < nblk; ++jb, ++g) {
        mbar_wait(smem_u32(&bars->s_full), g & 1);
        tc_fence_after();
        const int nch = block_chunks(Tv, jb);
        if (warp_active) {
          uint32_t v[16];
          if (jb == 0) {
            // exponent reference m' = floor(k2 * max of the first 16 columns of the row), a whole number of binades (key 0 is valid)
            tmem_ld16_nowait(lane_addr + kSCol, v);
            tmem_ld_wait();
            float mx = __uint_as_float(v[0]);
#pragma unroll
            for (int q = 1; q < 16; ++q)
              if (q < Tv) mx = fmaxf(mx, __uint_as_float(v[q]));
            mxk = floorf(mx * k2);
            mx_true = mx;
          }
          for (int ch = 0; ch < nch; ++ch) {
            const int c0 = jb * kTileRows + ch * 16;            // first key of the chunk
            if (jb != 0 || ch != 0) {
              tmem_ld16_nowait(lane_addr + kSCol + (uint32_t)(ch * 16), v);
              tmem_ld_wait();
            }
            const bool full = c0 + 16 <= Tv;
            float pj[16];
            if (kPol) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float4 p4 = *reinterpret_cast<const float4*>(&pol_s[c0 + 4 * q]);
                pj[4 * q] = p4.x; pj[4 * q + 1] = p4.y; pj[4 * q + 2] = p4.z; pj[4 * q + 3] = p4.w;
              }
              // the diagonal (mask 1 whatever the policy) lies in the chunks that overlap this warp's 32 rows: warp-uniform test
              if (c0 < qt * kTileRows + quad * 32 + 32 && c0 + 16 > qt * kTileRows + quad * 32) {
#pragma unroll
                for (int q = 0; q < 16; ++q)
                  if (c0 + q == i) pj[q] = 1.0f;
              }
            }
            float a[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              float e = ex2_approx(fmaf(__uint_as_float(v[q]), k2, -mxk));
              if (kPol) e *= pj[q];                              // keys past T: the policy row holds zeros there
              else if (!full && c0 + q >= Tv) e = 0.f;
              a[q] = e;
            }
            s0 += (a[0] + a[4]) + (a[8] + a[12]); s1 += (a[1] + a[5]) + (a[9] + a[13]);
            s2 += (a[2] + a[6]) + (a[10] + a[14]); s3 += (a[3] + a[7]) + (a[11] + a[15]);
            if (kPol) {
              // the true row maximum, masked keys included (the reference's eps terms follow it); off the critical path
              if (full) {
                const float m0 = fmax3(__uint_as_float(v[0]), __uint_as_float(v[1]), __uint_as_float(v[2]));
                const float m1 = fmax3(__uint_as_float(v[3]), __uint_as_float(v[4]), __uint_as_float(v[5]));
                const float m2 = fmax3(__uint_as_float(v[6]), __uint_as_float(v[7]), __uint_as_float(v[8]));
                const float m3 = fmax3(__uint_as_float(v[9]), __uint_as_float(v[10]), __uint_as_float(v[11]));
                const float m4 = fmax3(__uint_as_float(v[12]), __uint_as_float(v[13]), __uint_as_float(v[14]));
                mx_true = fmax3(mx_true, fmax3(m0, m1, m2), fmax3(m3, m4, __uint_as_float(v[15])));
              } else {
#pragma unroll
                for (int q = 0; q < 16; ++q)
                  if (c0 + q < Tv) mx_true = fmaxf(mx_true, __uint_as_float(v[q]));
              }
            }
            if (want_cls) {
#pragma unroll
              for (int q = 0; q < 16; ++q) cls_s[c0 + q] = a[q];
            }
            uint32_t packed[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) packed[q] = pack_bf16x2(a[2 * q], a[2 * q + 1]);
            if (ch == 0 && g > 0) {                             // P_{j-1} has been consumed by its PV-MMA
              mbar_wait(smem_u32(&bars->pv_done), (g - 1) & 1);
              tc_fence_after();
            }
            tmem_st8(lane_addr + kPCol + (uint32_t)(ch * 8), packed);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(smem_u32(&bars->p_full));
        if (kPol) {
          // colsum(V) over the valid keys of this block, for the eps/T term: 2 row groups x 64 columns
          const uint32_t st = g % kLongStages;
          mbar_wait(smem_u32(&bars->v_full[st]), (g / kLongStages) & 1);
          const int col = r & (kTcHD - 1), grp = r >> 6;
          const int rows = min(kTileRows, Tv - jb * kTileRows);
          const unsigned char* vb = v_s + st * kTileBytes;
          for (int j = grp; j < rows; j += 2)
            vacc += __bfloat162float(*(reinterpret_cast<const __nv_bfloat16*>(vb + sw128_off(j, col >> 3)) + (col & 7)));
          mbar_arrive(smem_u32(&bars->v_empty[st]));
        }
      }
      const uint32_t g_last = g - 1;
      if (kPol) {
        vpart_s[r] = vacc;
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (r < kTcHD) vsum_s[r] = vpart_s[r] + vpart_s[r + kTcHD];
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
      float sum = (s0 + s1) + (s2 + s3);
      // the one vote: a row holding a logit more than ~kMaxBinades above m' shows as a sum beyond 2^100, inf or NaN
      const bool fail = warp_active && i < Tv && !(sum <= kBigSum);
      float f = 1.0f;                                           // power of two applied to O, the sum and the CLS values
      if (kPol && warp_active && !fail) {
        // a MASKED key far above every kept one never shows in the sums; the reference still subtracts it, so m' follows it
        const float over = fmaf(mx_true, k2, -mxk);
        if (over > kMaxBinades) {
          const float d = floorf(over);
          f = exp2_neg_int(d);
          sum *= f;
          mxk += d;
        }
      }
      float eps_scale = (kPol && warp_active) ? ex2_approx(fmaf(mx_true, k2, -mxk)) : 1.0f;   // <= 2^kMaxBinades
      float den = sum + eps_den * eps_scale;
      float c_eps_row = c_eps * eps_scale;
      // ---- epilogue: O out of TMEM, normalised, straight to global memory ----
      mbar_wait(smem_u32(&bars->pv_done), g_last & 1);
      tc_fence_after();
      {
        const float inv = 1.0f / den;
        const bool store = warp_active && i < Tv && !fail;
        uint4* orow = reinterpret_cast<uint4*>(out + orow_off);
#pragma unroll
        for (int ch = 0; ch < kTcHD / 16; ++ch) {
          uint32_t v[16];
          tmem_ld16_nowait(lane_addr + kOCol + (uint32_t)(ch * 16), v);
          tmem_ld_wait();
          uint32_t ow[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float o0 = __uint_as_float(v[2 * q]) * f, o1 = __uint_as_float(v[2 * q + 1]) * f;
            if (kPol) {
              o0 += c_eps_row * vsum_s[ch * 16 + 2 * q];
              o1 += c_eps_row * vsum_s[ch * 16 + 2 * q + 1];
            }
            ow[q] = pack_bf16x2(o0 * inv, o1 * inv);
          }
          if (store) {
            orow[ch * 2] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
            orow[ch * 2 + 1] = make_uint4(ow[4], ow[5], ow[6], ow[7]);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(smem_u32(&bars->o_free));                     // the next unit's first PV-MMA may overwrite O
      if (fail) {
        // Rare (never seen on trained ViTs, but nothing forbids it): redo this row from the packed qkv in global memory in fp32,
        // over all valid keys: the true maximum first (reference = floor(k2 max), no overflow possible), then the exponentials
        // and the P V product, 16 output columns per pass.
        const uint4* qrow = reinterpret_cast<const uint4*>(qkv + ((size_t)b * T + i) * (size_t)(3 * H * kTcHD) + (size_t)h * kTcHD);
        const __nv_bfloat16* kbase = qkv + (size_t)b * T * (size_t)(3 * H * kTcHD) + (size_t)(H + h) * kTcHD;
        const __nv_bfloat16* vbase = kbase + (size_t)H * kTcHD;
        auto dot = [&](int j) -> float {
          const uint4* krow = reinterpret_cast<const uint4*>(kbase + (size_t)j * (size_t)(3 * H * kTcHD));
          float acc = 0.f;
#pragma unroll 1
          for (int wq = 0; wq < kTcHD / 8; ++wq) {
            const uint4 x = qrow[wq], y = krow[wq];
            acc = fmaf(bf16_lo(x.x), bf16_lo(y.x), acc); acc = fmaf(bf16_hi(x.x), bf16_hi(y.x), acc);
            acc = fmaf(bf16_lo(x.y), bf16_lo(y.y), acc); acc = fmaf(bf16_hi(x.y), bf16_hi(y.y), acc);
            acc = fmaf(bf16_lo(x.z), bf16_lo(y.z), acc); acc = fmaf(bf16_hi(x.z), bf16_hi(y.z), acc);
            acc = fmaf(bf16_lo(x.w), bf16_lo(y.w), acc); acc = fmaf(bf16_hi(x.w), bf16_hi(y.w), acc);
          }
          return acc;
        };
        float rmx = -INFINITY;
#pragma unroll 1
        for (int j = 0; j < Tv; ++j) rmx = fmaxf(rmx, dot(j));
        mxk = floorf(rmx * k2);
        mx_true = rmx;
        eps_scale = kPol ? ex2_approx(fmaf(mx_true, k2, -mxk)) : 1.0f;
        c_eps_row = c_eps * eps_scale;
        uint4* orow = reinterpret_cast<uint4*>(out + orow_off);
#pragma unroll 1
        for (int dc = 0; dc < kTcHD / 16; ++dc) {
          float acc[16];
#pragma unroll
          for (int q = 0; q < 16; ++q) acc[q] = 0.f;
          float rs = 0.f;
#pragma unroll 1
          for (int j = 0; j < Tv; ++j) {
            float e = ex2_approx(fmaf(dot(j), k2, -mxk));
            if (kPol && j != i) e *= pol_s[j];
            rs += e;
            if (dc == 0 && want_cls) cls_s[j] = e;
            const uint4* vrow = reinterpret_cast<const uint4*>(vbase + (size_t)j * (size_t)(3 * H * kTcHD) + dc * 16);
            const uint4 x0 = vrow[0], x1 = vrow[1];
            acc[0] = fmaf(e, bf16_lo(x0.x), acc[0]); acc[1] = fmaf(e, bf16_hi(x0.x), acc[1]);
            acc[2] = fmaf(e, bf16_lo(x0.y), acc[2]); acc[3] = fmaf(e, bf16_hi(x0.y), acc[3]);
            acc[4] = fmaf(e, bf16_lo(x0.z), acc[4]); acc[5] = fmaf(e, bf16_hi(x0.z), acc[5]);
            acc[6] = fmaf(e, bf16_lo(x0.w), acc[6]); acc[7] = fmaf(e, bf16_hi(x0.w), acc[7]);
            acc[8] = fmaf(e, bf16_lo(x1.x), acc[8]); acc[9] = fmaf(e, bf16_hi(x1.x), acc[9]);
            acc[10] = fmaf(e, bf16_lo(x1.y), acc[10]); acc[11] = fmaf(e, bf16_hi(x1.y), acc[11]);
            acc[12] = fmaf(e, bf16_lo(x1.z), acc[12]); acc[13] = fmaf(e, bf16_hi(x1.z), acc[13]);
            acc[14] = fmaf(e, bf16_lo(x1.w), acc[14]); acc[15] = fmaf(e, bf16_hi(x1.w), acc[15]);
          }
          den = rs + eps_den * eps_scale;
          const float inv = 1.0f / den;
          uint32_t ow[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float o0 = acc[2 * q], o1 = acc[2 * q + 1];
            if (kPol) {
              o0 += c_eps_row * vsum_s[dc * 16 + 2 * q];
              o1 += c_eps_row * vsum_s[dc * 16 + 2 * q + 1];
            }
            ow[q] = pack_bf16x2(o0 * inv, o1 * inv);
          }
          orow[dc * 2] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
          orow[dc * 2 + 1] = make_uint4(ow[4], ow[5], ow[6], ow[7]);
        }
        f = 1.0f;
      }
      if (cls_dst != nullptr && qt == 0 && warp == 0) {
        // CLS row (query 0 = lane 0 of warp 0): probabilities of row 0, Attention.forward's second output
        __syncwarp();
        const float den0 = __shfl_sync(0xffffffffu, den, 0);
        const float ce0 = __shfl_sync(0xffffffffu, c_eps_row, 0);
        const float f0 = __shfl_sync(0xffffffffu, f, 0);
        for (int j = lane; j < T; j += 32) cls_dst[j] = j < Tv ? (cls_s[j] * f0 + ce0) / den0 : 0.f;
        __syncwarp();
      }
      if (kVar && i >= Tv && i < T) {                           // pad rows of the output: zeros
        uint4* orow = reinterpret_cast<uint4*>(out + orow_off);
#pragma unroll
        for (int q = 0; q < kTcHD / 8; ++q) orow[q] = make_uint4(0u, 0u, 0u, 0u);
      }
      ++un;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kLongMmaWarp) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(kLongTmemCols) : "memory");
  }
}

template <bool kPol, bool kVar>
int launch_long(const CUtensorMap& map, const float* policy, const int* lens, int units, LongShape shp, float scale, float eps,
                void* out, float* cls_row, const void* qkv, cudaStream_t stream) {
  auto kern = attn_long_fwd_kernel<kPol, kVar>;
  static SmemOptIn opt;  // one per instantiation
  cudaError_t e = opt_in_smem(opt, kern, (int)kLongSmem);
  D2S_REQUIRE(e == cudaSuccess, D2S_ERR_CUDA, "attn_long_fwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  const int grid = units < 2 * kNumSMs ? units : 2 * kNumSMs;
  kern<<<grid, kLongThreads, kLongSmem, stream>>>(map, policy, lens, units, shp, scale, eps, (__nv_bfloat16*)out, cls_row,
                                                 (const __nv_bfloat16*)qkv);
  count_launch();
  return check_launch("d2s_attn_long_fwd(tcgen05)");
}

}  // namespace
}  // namespace d2s

using namespace d2s;

extern "C" int d2s_attn_long_fwd(const void* qkv, const float* policy, const int* len, int B, int T, int H, int hd, float scale,
                                 float eps, void* out, float* cls_row, d2s_stream_t stream_) {
  D2S_REQUIRE(qkv && out, D2S_ERR_ARG, "attn_long_fwd: null pointer");
  D2S_REQUIRE(hd == kTcHD, D2S_ERR_ARG, "attn_long_fwd: head dim %d unsupported (64 only)", hd);
  D2S_REQUIRE(B >= 0 && H >= 1 && T >= 1 && T <= kLongMaxT, D2S_ERR_ARG, "attn_long_fwd: bad shape B=%d T=%d H=%d (1 <= T <= %d)",
              B, T, H, kLongMaxT);
  D2S_REQUIRE(!(policy && len), D2S_ERR_ARG, "attn_long_fwd: policy and len are exclusive (the variable-length form takes no policy)");
  const int nqt = ceil_div(T, kTileRows);
  D2S_REQUIRE((long long)B * H * nqt <= (1LL << 30), D2S_ERR_ARG, "attn_long_fwd: B*H=%lld too large", (long long)B * H);
  D2S_REQUIRE(scale > 0.0f, D2S_ERR_ARG, "attn_long_fwd: scale must be positive (got %g)", (double)scale);
  D2S_REQUIRE(aligned16(qkv) && aligned16(out), D2S_ERR_ALIGN, "attn_long_fwd: qkv/out must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  EncodeFn enc = encode_fn();
  D2S_REQUIRE(enc != nullptr, D2S_ERR_CUDA, "attn_long_fwd: cuTensorMapEncodeTiled is unavailable from the driver");
  // 3-D view of the packed qkv buffer: (3*H*64 columns, T tokens, B images), box 64 x 128 rows; rows past T are zero-filled
  CUtensorMap map;
  const cuuint64_t gdim[3] = {(cuuint64_t)3 * H * kTcHD, (cuuint64_t)T, (cuuint64_t)B};
  const cuuint64_t gstride[2] = {(cuuint64_t)3 * H * kTcHD * 2, (cuuint64_t)T * 3 * H * kTcHD * 2};
  const cuuint32_t box[3] = {(cuuint32_t)kTcHD, (cuuint32_t)kTileRows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult cr = enc(&map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(qkv), gdim, gstride, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  D2S_REQUIRE(cr == CUDA_SUCCESS, D2S_ERR_CUDA, "attn_long_fwd: cuTensorMapEncodeTiled failed (%d)", (int)cr);
  cudaStream_t stream = (cudaStream_t)stream_;
  const LongShape shp{T, H, nqt};
  const int units = B * H * nqt;
  if (len) return launch_long<false, true>(map, nullptr, len, units, shp, scale, 0.0f, out, cls_row, qkv, stream);
  if (policy) return launch_long<true, false>(map, policy, nullptr, units, shp, scale, eps, out, cls_row, qkv, stream);
  return launch_long<false, false>(map, nullptr, nullptr, units, shp, scale, eps, out, cls_row, qkv, stream);
}
