// Kernel family (4), tensor-core part: policy-masked attention on tcgen05 / TMEM (bf16 in, fp32 accumulate).
//
//   S = Q K^T        tcgen05.mma kind::f16, A = Q tile (128 x 64, K-major, SWIZZLE_128B smem),
//                    B = K (Tkp x 64, K-major, SWIZZLE_128B smem), D = S in TMEM (128 lanes x Tkp cols fp32)
//   P = policy softmax, one query row per thread straight out of TMEM (tcgen05.ld 32x32b), unnormalised
//                    a_ij = exp((s_ij - max_j s_ij) * scale) * m_ij written back to TMEM as packed bf16
//                    over the dead S columns (tcgen05.st), row sums kept in registers
//   O = P V          tcgen05.mma with A = P from TMEM, B = V (MN-major SWIZZLE_128B smem), D = O in TMEM
//   out = (O + (eps/T) * colsum(V)) / (rowsum + eps)     -- the reference's "+eps/T on every entry" term
//                    (vit_models/dynamic_vit.py:213) folded into one per-head vector; CLS row side output.
//
// Execution model: persistent CTAs (2 per SM for T > 128, 4 per SM for T <= 128), each looping over (image, head)
// units.  Warp 4 lane 0 is the control thread: it issues the TMA loads (one 3-D tensor map over the packed
// (B, T, 3*H*64) qkv buffer, box = 64 x 128 rows, SWIZZLE_128B, rows past T zero-filled by the TMA unit) and the
// tcgen05.mma instructions; warps 0-3 are the softmax/epilogue warps (TMEM lane quadrant = warp id).  Inside one
// CTA a unit is a serial chain S-MMA -> softmax -> PV-MMA -> epilogue; the loads of the NEXT unit are issued as soon
// as their buffers die (Q/K after the last S-MMA, V after the last PV-MMA) so they land during the softmax, and the
// other CTAs resident on the SM fill the tensor / MUFU / FMA pipes while this one waits.
//
// Per image-layer (T=197, H=6): 59.6 MFLOP against 611 KB of algorithmic HBM traffic (SURVEY.md 8d): HBM-bound
// unless the QKV projection is fused; the scores never touch HBM.  The MUFU (exp2) floor is ~64 us for B=1024.
#pragma once
#include "d2s_tc.cuh"

namespace d2s {

// warps [0, kSW): softmax/epilogue (TMEM lane quadrant = warp % 4; with kSW == 8 the two warps of a quadrant split the
// key columns of every row); warp kSW: TMA + MMA issue
constexpr int tc_threads(int ksw) { return 32 * (ksw + 1); }
// a logit this many binades (powers of two, after scaling) above the row's exponent reference raises the reference
constexpr float kMaxBinades = 100.0f;
constexpr float kBigSum = 1.2676506e30f;   // 2^100: a row whose partial sums end beyond it (or inf, or NaN) is redone with its true maximum

// clock64 wait / phase totals per CTA (profiling builds only: D2S_NVCC_EXTRA=-DD2S_ATTN_TRACE_BUILD; scripts/bench_attn_trace.py)
#ifdef D2S_ATTN_TRACE_BUILD
__device__ long long d2s_tc_trace_buf[1024 * 16];
#define TC_TRACE_DECL long long tr[8] = {}; long long tr_t = clock64(); const long long tr_begin = tr_t;
#define TC_TRACE(i) { const long long tr_n = clock64(); tr[i] += tr_n - tr_t; tr_t = tr_n; }
#define TC_TRACE_DUMP(slot) if (lane == 0 && blockIdx.x < 1024) { long long* dst = d2s_tc_trace_buf + (size_t)blockIdx.x * 16 + (slot) * 8; \
    for (int i = 0; i < 7; ++i) dst[i] = tr[i]; dst[7] = clock64() - tr_begin; }
#else
#define TC_TRACE_DECL
#define TC_TRACE(i)
#define TC_TRACE_DUMP(slot)
#endif

struct TcBars {
  uint64_t q_full[2], k_full[2], v_full, s_full, p_full, o_full, tmem_free;
  uint32_t tmem_base;
  uint32_t pad;
};

// Valid tokens of image b in the variable-length form (d2s_attn_varlen_fwd): lens[b] clamped to [0, T], T = the padded length
__device__ __forceinline__ int var_len(const int* __restrict__ lens, int b, int T) { return min(max(lens[b], 0), T); }
// 16-column key chunks a unit of the variable-length form runs (softmax, P columns, PV K-steps): those holding its valid keys.  With
// two softmax warps per row at least 3, so that the first column half's P (columns [0, 8 ceil(n/2))) stays below the shared
// reference chunk ceil(n/2) - 1 that the second half reads.  Equals the dense kernel's Tkp / 16 at T = lens[b].
__device__ __forceinline__ int var_chunks(int Tv, int ksw) { return max((Tv + 15) >> 4, ksw == 8 ? 3 : 1); }

// kNT  : 128-row tiles per unit (1: T <= 128, 2: T <= 256)
// kPol : policy given (eps terms, masked exponentials, colsum(V))
// kVar : variable-length form: image b has Tv = lens[b] valid tokens of the T (padded) rows; keys, query rows, votes and the rare
//        path follow Tv, output rows and cls_row columns Tv..T-1 are written as zeros (no policy, no stats)
template <int kNT, bool kPol, int kSW, bool kVar = false>
__global__ void __launch_bounds__(tc_threads(kSW), kNT == 1 ? 4 : 2)
attn_tc_fwd_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                   const float* __restrict__ policy, int num_units, int T, int H, int Tkp, int kbufs, float scale,
                   float eps, __nv_bfloat16* __restrict__ out, float* __restrict__ cls_row, float* __restrict__ stats,
                   const __nv_bfloat16* __restrict__ qkv, const int* __restrict__ lens) {
  static_assert(!(kVar && kPol), "the variable-length form takes no policy");
  constexpr int kTmemCols = kNT == 1 ? 128 : 256;
  // O accumulator columns: beyond the packed-P columns.  One softmax warp per row: P at [0, Tkp/2).  Two warps per row
  // (kSW == 8): the second column half writes its P over ITS OWN consumed S columns, at [16*ceil(n/2), ...) <= 192.
  constexpr int kOCol = kNT == 1 ? 64 : (kSW == 8 ? 192 : 128);
  extern __shared__ unsigned char smem_dyn[];
  // SWIZZLE_128B atoms are 1024 B and address based: align the tile region.  Every buffer is a whole number of
  // 8-row atoms.  rows_a = rows of the first TMA box (map_a), rows_b = rows of the second one (map_b, kNT == 2).
  const int rows_a = kNT == 1 ? Tkp : kTileRows;
  const int rows_b = kNT == 1 ? 0 : Tkp - kTileRows;
  const uint32_t raw = smem_u32(smem_dyn);
  const uint32_t pad = (1024u - (raw & 1023u)) & 1023u;
  unsigned char* tiles = smem_dyn + pad;
  unsigned char* q_s[2];
  q_s[0] = tiles;                                             // 128 x 128 B (the MMA always reads 128 rows)
  q_s[1] = q_s[0] + kTileBytes;                               // rows_b x 128 B (the MMA reads 128 rows: the tail rows
                                                              // alias the K buffer and only feed query rows >= T)
  unsigned char* k_s0 = q_s[1] + rows_b * 128;                // kbufs x (Tkp x 128 B)
  unsigned char* v_s = k_s0 + (size_t)kbufs * Tkp * 128;      // Tkp x 128 B
  TcBars* bars = reinterpret_cast<TcBars*>(v_s + (size_t)Tkp * 128);
  float* pol_s = reinterpret_cast<float*>(bars + 1);          // 256
  float* cls_s = pol_s + 256;                                 // 256
  float* vsum_s = cls_s + 256;                                // 64
  float* sum_s = vsum_s + 64;                                 // 2 x 128 (kSW == 8: partial row sums of the column halves)
  float* max_s = sum_s + 256;                                 // 2 x 128
  float* ref_s = max_s + 256;                                 // 2 x 128 (kSW == 8: exponent reference of each column half)
  float* vpart_s = ref_s + 256;                               // 4 x 64 partial column sums of V

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t bytes_a = (uint32_t)rows_a * 128u, bytes_b = (uint32_t)rows_b * 128u;

  if (tid == 0) {
    mbar_init(smem_u32(&bars->q_full[0]), 1);
    mbar_init(smem_u32(&bars->q_full[1]), 1);
    mbar_init(smem_u32(&bars->k_full[0]), 1);
    mbar_init(smem_u32(&bars->k_full[1]), 1);
    mbar_init(smem_u32(&bars->v_full), 1);
    mbar_init(smem_u32(&bars->s_full), 1);
    mbar_init(smem_u32(&bars->p_full), 32 * kSW);
    mbar_init(smem_u32(&bars->o_full), 1);
    mbar_init(smem_u32(&bars->tmem_free), 32 * kSW);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kSW) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)),
                 "n"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;

  if (warp_uniform(warp) == kSW) {
    {
      // ====== control warp: TMA + MMA issue.  The whole warp runs the loop warp-uniformly (waits, address arithmetic) and one
      // elected lane issues each TMA / tcgen05 instruction: under `if (lane == 0)` every tcgen05.mma was wrapped in an
      // ELECT / R2UR.BROADCAST waterfall loop (72-cycle issue cadence against 32 cycles of tensor work per PV step) ======
      const uint32_t idesc_s = make_idesc(128, Tkp, 0);
      const uint32_t idesc_o = make_idesc(128, kTcHD, 1);
      const uint64_t vd = make_desc_sw128(smem_u32(v_s), 16, 1024);
      const int ksteps = Tkp / 16;
      // one operand = one box of rows_a rows (+ one of rows_b rows), landing contiguously
      auto load_rows = [&](unsigned char* dst, int col, int b, uint32_t bar) {
        if (elect_one()) {
          mbar_expect_tx(bar, bytes_a + bytes_b);
          tma_load_3d(smem_u32(dst), &map_a, col, 0, b, bar);
          if (kNT == 2) tma_load_3d(smem_u32(dst) + bytes_a, &map_b, col, kTileRows, b, bar);
        }
        __syncwarp();
      };
      auto issue_k = [&](int unit, uint32_t it) {
        const uint32_t kb = kbufs == 2 ? (it & 1) : 0;
        load_rows(k_s0 + (size_t)kb * Tkp * 128, (H + unit % H) * kTcHD, unit / H, smem_u32(&bars->k_full[kb]));
      };
      auto issue_q = [&](int unit, int t) {
        const uint32_t bar = smem_u32(&bars->q_full[t]);
        if (elect_one()) {
          mbar_expect_tx(bar, t == 0 ? bytes_a : bytes_b);
          tma_load_3d(smem_u32(q_s[t]), t == 0 ? &map_a : &map_b, (unit % H) * kTcHD, t * kTileRows, unit / H, bar);
        }
        __syncwarp();
      };
      auto issue_v = [&](int unit) { load_rows(v_s, (2 * H + unit % H) * kTcHD, unit / H, smem_u32(&bars->v_full)); };
      int unit = blockIdx.x;
      if (unit < num_units) {
        issue_k(unit, 0);
#pragma unroll
        for (int t = 0; t < kNT; ++t) issue_q(unit, t);
        issue_v(unit);
      }
      uint32_t g = 0;  // tiles processed by this CTA: parity source for the per-tile barriers
      TC_TRACE_DECL
      for (uint32_t it = 0; unit < num_units; unit += gridDim.x, ++it) {
        const int next = unit + gridDim.x;
        const bool has_next = next < num_units;
        const uint32_t kb = kbufs == 2 ? (it & 1) : 0;
        const uint32_t k_parity = kbufs == 2 ? ((it >> 1) & 1) : (it & 1);
        const int ks_u = kVar ? var_chunks(var_len(lens, unit / H, T), kSW) : ksteps;
        // with two K buffers the next unit's K is requested a whole unit ahead (its buffer died one unit ago)
        if (kbufs == 2 && has_next) issue_k(next, it + 1);
        const uint64_t kd = make_desc_sw128(smem_u32(k_s0 + (size_t)kb * Tkp * 128), 16, 1024);
#pragma unroll
        for (int t = 0; t < kNT; ++t, ++g) {
          TC_TRACE(6)
          if (t == 0) mbar_wait(smem_u32(&bars->k_full[kb]), k_parity);
          TC_TRACE(0)
          mbar_wait(smem_u32(&bars->q_full[t]), it & 1);
          TC_TRACE(1)
          if (g > 0) mbar_wait(smem_u32(&bars->tmem_free), (g - 1) & 1);
          TC_TRACE(2)
          tc_fence_after();
          const uint64_t qd = make_desc_sw128(smem_u32(q_s[t]), 16, 1024);
          if (elect_one()) {
            mma_ss_imm<false>(tmem, qd, kd, idesc_s);
            mma_ss_imm<true>(tmem, qd + 2, kd + 2, idesc_s);
            mma_ss_imm<true>(tmem, qd + 4, kd + 4, idesc_s);
            mma_ss_imm<true>(tmem, qd + 6, kd + 6, idesc_s);
            mma_commit(smem_u32(&bars->s_full));
          }
          __syncwarp();
          const bool last = t == kNT - 1;
          TC_TRACE(6)
          mbar_wait(smem_u32(&bars->p_full), g & 1);   // softmax done => this tile's S-MMA has completed as well
          TC_TRACE(3)
          if (has_next) {
            issue_q(next, t);                          // this Q tile is dead: refill it during PV / epilogue / softmax
            if (last && kbufs == 1) issue_k(next, it + 1);
          }
          TC_TRACE(6)
          if (t == 0) mbar_wait(smem_u32(&bars->v_full), it & 1);
          TC_TRACE(4)
          tc_fence_after();
          // fully unrolled issue (T <= 256 => at most 16 K-steps); descriptors advance by constants
          const int split = kSW == 8 ? (ks_u + 1) / 2 : 16;     // first K-step whose P lives in the second half's region
          if (elect_one()) {
            mma_ts_imm<false>(tmem + kOCol, tmem, vd, idesc_o);
#pragma unroll
            for (int ks = 1; ks < 16; ++ks)
              if (ks < ks_u) {
                const uint32_t pa = ks < split ? (uint32_t)(ks * 8) : (uint32_t)(split * 16 + (ks - split) * 8);
                mma_ts_imm<true>(tmem + kOCol, tmem + pa, vd + (uint64_t)(ks * 128), idesc_o);
              }
            mma_commit(smem_u32(&bars->o_full));
          }
          __syncwarp();
          if (last && has_next) {
            TC_TRACE(6)
            mbar_wait(smem_u32(&bars->o_full), g & 1);  // V is dead once the PV-MMA has completed
            TC_TRACE(5)
            issue_v(next);
          }
        }
      }
      TC_TRACE(6)
      TC_TRACE_DUMP(0)
    }
  } else {
    // ===================================== softmax / epilogue warps =====================================
    const int quad = warp & 3, half = warp >> 2;   // TMEM lane quadrant; column half (kSW == 8 only)
    const int r = quad * 32 + lane;                // row inside the tile == TMEM lane
    const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16);
    const float k2 = scale * 1.4426950408889634f;
    const float c_eps = kPol ? eps / (float)T : 0.0f;
    const float eps_den = kPol ? eps : 0.0f;
    const int nchunks = Tkp / 16;
    uint32_t g = 0;
    constexpr int kPolPer = 256 / (32 * kSW);                     // policy elements per softmax thread (256-entry row buffer)
    float pol_next[kPolPer];
    TC_TRACE_DECL
    for (uint32_t it = 0, unit = blockIdx.x; (int)unit < num_units; unit += gridDim.x, ++it) {
      const int b = unit / H, h = unit % H;
      const int Tv = kVar ? var_len(lens, b, T) : T;               // valid tokens of this image
      const int nch = kVar ? var_chunks(Tv, kSW) : nchunks;
      if (kPol) {
        // per-unit policy row and column sums of V (for the eps/T term): sum_j V[j][d].  The policy row of THIS unit was fetched
        // into registers while the previous unit was being processed (its global-memory latency is off the critical path); the
        // column sums are split over all softmax threads (row groups x 64 columns) and combined through shared memory.
        asm volatile("bar.sync 1, %0;" ::"n"(32 * kSW) : "memory");  // previous unit's readers of pol_s / vsum_s are done
        if (it == 0) {
#pragma unroll
          for (int q = 0; q < kPolPer; ++q) {
            const int j = tid + q * 32 * kSW;
            pol_next[q] = (j < T) ? policy[(size_t)b * T + j] : 0.0f;
          }
        }
#pragma unroll
        for (int q = 0; q < kPolPer; ++q) pol_s[tid + q * 32 * kSW] = pol_next[q];
        {
          const int nb = (int)(unit + gridDim.x) / H;             // next unit's image (clamped: the values are unused past the end)
          const int nbc = nb < (num_units / H) ? nb : b;
#pragma unroll
          for (int q = 0; q < kPolPer; ++q) {
            const int j = tid + q * 32 * kSW;
            pol_next[q] = (j < T) ? policy[(size_t)nbc * T + j] : 0.0f;
          }
        }
        mbar_wait(smem_u32(&bars->v_full), it & 1);
        {
          constexpr int kGroups = 32 * kSW / kTcHD;               // row groups: 2 (four softmax warps) or 4 (eight)
          const int col = tid & (kTcHD - 1), grp = tid >> 6;
          const int cchunk = col >> 3, within = col & 7;
          float acc = 0.f;
          for (int j = grp; j < T; j += kGroups)
            acc += __bfloat162float(*(reinterpret_cast<const __nv_bfloat16*>(v_s + sw128_off(j, cchunk)) + within));
          vpart_s[grp * kTcHD + col] = acc;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(32 * kSW) : "memory");
        if (tid < kTcHD) {
          constexpr int kGroups = 32 * kSW / kTcHD;
          float acc = vpart_s[tid];
#pragma unroll
          for (int gq = 1; gq < kGroups; ++gq) acc += vpart_s[gq * kTcHD + tid];
          vsum_s[tid] = acc;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(32 * kSW) : "memory");
      }
#pragma unroll
      for (int t = 0; t < kNT; ++t, ++g) {
        const int i = t * kTileRows + r;                  // query token of this thread
        const bool warp_active = t * kTileRows + quad * 32 < Tv;  // whole warp beyond T: nothing to compute
        // key columns of this warp: all of them (kSW == 4) or one half, split at a 16-column chunk boundary
        const int ch_lo = (kSW == 8 && half == 1) ? (nch + 1) / 2 : 0;
        const int ch_hi = (kSW == 8 && half == 0) ? (nch + 1) / 2 : nch;
        TC_TRACE(6)
        mbar_wait(smem_u32(&bars->s_full), g & 1);
        TC_TRACE(0)
        tc_fence_after();
        float sum = 0.f, mx_true = -INFINITY, mxk = 0.f;
        const bool want_cls = (cls_row != nullptr) && (i == 0);
        // TMEM column of the packed-P chunk `c` of this warp (second column half: its own region, see kOCol)
        auto pcol = [&](int c) -> uint32_t {
          return (kSW == 8 && half == 1) ? (uint32_t)(ch_lo * 16 + (c - ch_lo) * 8) : (uint32_t)(c * 8);
        };
        // Multiply everything this thread has produced for chunks [ch_lo, upto) by f = 2^-d (exact: P is bf16, f a power of
        // two).  Warp-uniform call (tcgen05.ld/st are .sync.aligned), per-lane f.
        auto rescale_row = [&](int upto, float f, float& s0, float& s1, float& s2, float& s3) {
          s0 *= f; s1 *= f; s2 *= f; s3 *= f;
          tmem_st_wait();
          for (int c = ch_lo; c < upto; ++c) {
            uint32_t w[8];
            tmem_ld8_nowait(lane_addr + pcol(c), w);
            tmem_ld_wait();
#pragma unroll
            for (int q = 0; q < 8; ++q) w[q] = pack_bf16x2(bf16_lo(w[q]) * f, bf16_hi(w[q]) * f);
            tmem_st8(lane_addr + pcol(c), w);
          }
          if (want_cls)
            for (int j = ch_lo * 16; j < upto * 16; ++j) cls_s[j] *= f;
        };
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        if (warp_active) {
          // ONE pass over S (reading S twice -- row max, then exponentials -- lengthens the serial chain of the tile).
          // Exponentials are taken against a reference m' = floor(k2 * max of 16 columns of the row), not the row max: softmax
          // is shift invariant and bf16 keeps fp32's exponent range, so P = 2^(k2 s - m') is as accurate as 2^(k2 (s - max)).
          // The true max is tracked on the side because the reference's eps terms are not shift invariant; they are rescaled
          // by 2^(k2 max - m') below, which restores the reference formula exactly.  m' is an INTEGER number of binades, so that
          // it can be raised after the fact by multiplying what was produced with a power of two (exact): the masked-key case
          // and the two-warps-per-row reconciliation below.  A row holding a logit more than kMaxBinades above m' (never seen on
          // trained ViTs, but nothing forbids it) is found by ONE test of its finished partial sums after the loop and redone
          // from global memory with its true maximum as the reference, so the result does not depend on where the maximum sits.
          // Reference chunk: chunk 0 with one warp per row.  With two warps per row both must derive the SAME m' from
          // columns neither of them overwrites with P before the other has read them: the last chunk of the first
          // half (the first half's P ends at column 8*ceil(n/2), below that chunk; the second half's P starts above it).
          const int ch_ref = kSW == 8 ? (nch + 1) / 2 - 1 : 0;
          uint32_t v[16];
          tmem_ld16_nowait(lane_addr + (uint32_t)(ch_ref * 16), v);
          tmem_ld_wait();
          // (variable-length form: a short image in a two-tile batch may have no valid key in the shared reference chunk; its rows
          // then start from -inf, overflow at once and are redone by the rare path below, never reading a pad column)
          float mx = (kVar && ch_ref * 16 >= Tv) ? -INFINITY : __uint_as_float(v[0]);
#pragma unroll
          for (int q = 1; q < 16; ++q)
            if (ch_ref * 16 + q < Tv) mx = fmaxf(mx, __uint_as_float(v[q]));
          mxk = floorf(mx * k2);
          mx_true = mx;
          // exponentials of S chunk `c` (in `src`) against the current reference, times the policy.  The diagonal (mask 1 whatever
          // the policy) lies in the chunks that overlap this warp's 32 query rows: a warp-uniform split, so that every other chunk is
          // a plain multiply by the policy (fetched as four 16-byte broadcasts)
          auto exps_of = [&](const uint32_t (&src)[16], int c, float (&dst)[16]) {
            const bool cfull = c * 16 + 16 <= Tv;
            float pj[16];
            if (kPol) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float4 p4 = *reinterpret_cast<const float4*>(&pol_s[c * 16 + 4 * q]);
                pj[4 * q] = p4.x; pj[4 * q + 1] = p4.y; pj[4 * q + 2] = p4.z; pj[4 * q + 3] = p4.w;
              }
              if (c * 16 < t * kTileRows + quad * 32 + 32 && c * 16 + 16 > t * kTileRows + quad * 32) {
#pragma unroll
                for (int q = 0; q < 16; ++q)
                  if (c * 16 + q == i) pj[q] = 1.0f;
              }
            }
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              float e = ex2_approx(fmaf(__uint_as_float(src[q]), k2, -mxk));
              if (kPol) e *= pj[q];                       // columns past T: the policy buffer holds zeros there
              else if (!cfull && c * 16 + q >= Tv) e = 0.f;
              dst[q] = e;
            }
          };
          // The chunk loop carries NO overflow handling: a logit more than 128 binades above the reference simply turns into inf
          // (or NaN under a zero policy) and shows in the row's partial sums, which are tested ONCE after the loop (a vote and a
          // branch inside the loop, between a chunk's last exponential and its tcgen05.st, cost 14 % of the kernel at T = 197 and
          // more below, profiles/r02zz_attn_overflow_check.txt).
          for (int ch = ch_lo; ch < ch_hi; ++ch) {
            TC_TRACE(6)
            if (ch != ch_ref || ch != ch_lo) {   // (the reference chunk is still in registers only if it comes first)
              tmem_ld16_nowait(lane_addr + (uint32_t)(ch * 16), v);
              tmem_ld_wait();
            }
            TC_TRACE(1)
            float a[16];
            const bool full = ch * 16 + 16 <= Tv;
            exps_of(v, ch, a);
            s0 += (a[0] + a[4]) + (a[8] + a[12]); s1 += (a[1] + a[5]) + (a[9] + a[13]);
            s2 += (a[2] + a[6]) + (a[10] + a[14]); s3 += (a[3] + a[7]) + (a[11] + a[15]);
            if (kPol) {
              // the true row maximum (masked keys included: the reference's eps terms follow it); off the critical path
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
                  if (ch * 16 + q < Tv) mx_true = fmaxf(mx_true, __uint_as_float(v[q]));
              }
            }
            if (want_cls) {
#pragma unroll
              for (int q = 0; q < 16; ++q) cls_s[ch * 16 + q] = a[q];
            }
            TC_TRACE(5)
            uint32_t packed[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) packed[q] = pack_bf16x2(a[2 * q], a[2 * q + 1]);
            // P overlays S columns this warp has already consumed
            tmem_st8(lane_addr + pcol(ch), packed);
            TC_TRACE(2)
          }
          // (rows past T take no part in the votes: inside the last 16-row granule they are zero-filled by TMA, beyond it the MMA
          // reads shared memory nobody wrote, and a NaN there would send the whole warp down the rare paths for nothing)
          if (__any_sync(0xffffffffu, i < Tv && !((s0 + s1) + (s2 + s3) <= kBigSum))) {
            // Rare (never seen on trained ViTs, but nothing forbids it): a row of this warp holds a logit more than kMaxBinades
            // above its reference (a partial sum beyond 2^kMaxBinades, inf or NaN).  S is gone by now -- P overlays it -- so the
            // warp redoes its 32 rows from the packed qkv in global memory, two passes: fp32 dot products q_i . k_j for the row
            // maximum over this warp's key columns, reference = floor(k2 max) (no overflow possible), then the exponentials.  With
            // two warps per row the halves may now end on different references; the exchange below reconciles them (exact).
            const int iq = i < Tv ? i : Tv - 1;
            const uint4* qrow = reinterpret_cast<const uint4*>(qkv + ((size_t)b * T + iq) * (size_t)(3 * H * kTcHD) + (size_t)h * kTcHD);
            const __nv_bfloat16* kbase = qkv + (size_t)b * T * (size_t)(3 * H * kTcHD) + (size_t)(H + h) * kTcHD;
            auto dot = [&](int j) -> float {
              const uint4* krow = reinterpret_cast<const uint4*>(kbase + (size_t)j * (size_t)(3 * H * kTcHD));
              float acc = 0.f;
#pragma unroll 1
              for (int w = 0; w < kTcHD / 8; ++w) {
                const uint4 x = qrow[w], y = krow[w];
                acc = fmaf(bf16_lo(x.x), bf16_lo(y.x), acc); acc = fmaf(bf16_hi(x.x), bf16_hi(y.x), acc);
                acc = fmaf(bf16_lo(x.y), bf16_lo(y.y), acc); acc = fmaf(bf16_hi(x.y), bf16_hi(y.y), acc);
                acc = fmaf(bf16_lo(x.z), bf16_lo(y.z), acc); acc = fmaf(bf16_hi(x.z), bf16_hi(y.z), acc);
                acc = fmaf(bf16_lo(x.w), bf16_lo(y.w), acc); acc = fmaf(bf16_hi(x.w), bf16_hi(y.w), acc);
              }
              return acc;
            };
            const int j_hi = ch_hi * 16 < Tv ? ch_hi * 16 : Tv;
            float rmx = -INFINITY;
#pragma unroll 1
            for (int j = ch_lo * 16; j < j_hi; ++j) rmx = fmaxf(rmx, dot(j));
            mxk = floorf(rmx * k2);
            mx_true = rmx;
            s0 = s1 = s2 = s3 = 0.f;
            tmem_st_wait();
#pragma unroll 1
            for (int c = ch_lo; c < ch_hi; ++c) {
              uint32_t u[16];
#pragma unroll 1
              for (int q = 0; q < 16; ++q) u[q] = __float_as_uint(c * 16 + q < Tv ? dot(c * 16 + q) : 0.f);
              float e16[16];
              exps_of(u, c, e16);
              s0 += (e16[0] + e16[4]) + (e16[8] + e16[12]); s1 += (e16[1] + e16[5]) + (e16[9] + e16[13]);
              s2 += (e16[2] + e16[6]) + (e16[10] + e16[14]); s3 += (e16[3] + e16[7]) + (e16[11] + e16[15]);
              if (want_cls) {
#pragma unroll
                for (int q = 0; q < 16; ++q) cls_s[c * 16 + q] = e16[q];
              }
              uint32_t w8[8];
#pragma unroll
              for (int q = 0; q < 8; ++q) w8[q] = pack_bf16x2(e16[2 * q], e16[2 * q + 1]);
              tmem_st8(lane_addr + pcol(c), w8);
            }
          }
          if (kPol) {
            // a MASKED key far above every kept one never shows in the sums: the reference still subtracts it (its row then
            // degenerates to the eps terms), so the reference is raised for it as well
            const float over = fmaf(mx_true, k2, -mxk);
            if (__any_sync(0xffffffffu, i < Tv && over > kMaxBinades)) {
              const float d = over > kMaxBinades ? floorf(over) : 0.f;
              rescale_row(ch_hi, exp2_neg_int(d), s0, s1, s2, s3);
              mxk += d;
            }
          }
        }  // rows of an idle warp are never written out; whatever their P rows hold stays in those rows
        if constexpr (kSW == 8) {
          // The two column halves of a row exchange their partial sums, running maxima and exponent references through shared
          // memory BEFORE P is published: both halves of a row must end on the same reference (one PV product reads both).
          sum_s[half * kTileRows + r] = (s0 + s1) + (s2 + s3);
          max_s[half * kTileRows + r] = mx_true;
          ref_s[half * kTileRows + r] = mxk;
          asm volatile("bar.sync %0, 64;" ::"r"(3 + quad) : "memory");        // the two warps of this row quadrant
          const float o_ref = ref_s[(half ^ 1) * kTileRows + r];
          float o_sum = sum_s[(half ^ 1) * kTileRows + r];
          if (__any_sync(0xffffffffu, warp_active && i < Tv && o_ref != mxk)) {  // rare: one half raised its reference
            const float d = warp_active ? fmaxf(o_ref - mxk, 0.f) : 0.f;   // integer: both started from the same m'
            if (warp_active) o_sum *= exp2_neg_int(fmaxf(mxk - o_ref, 0.f));
            rescale_row(ch_hi, exp2_neg_int(d), s0, s1, s2, s3);
            mxk += d;
            // (the branch is taken by both warps of a row pair or by neither: the partner's CLS-row share is final after this)
            asm volatile("bar.sync %0, 64;" ::"r"(7 + quad) : "memory");
          }
          sum = (s0 + s1) + (s2 + s3) + o_sum;
          if (kPol) mx_true = fmaxf(mx_true, max_s[(half ^ 1) * kTileRows + r]);
        } else {
          sum = (s0 + s1) + (s2 + s3);
        }
        TC_TRACE(6)
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        mbar_arrive(smem_u32(&bars->p_full));
        TC_TRACE(2)
        const float eps_scale = (kPol && warp_active) ? ex2_approx(fmaf(mx_true, k2, -mxk)) : 1.0f;   // <= 2^kMaxBinades
        const float den = sum + eps_den * eps_scale;
        const float c_eps_row = c_eps * eps_scale;
        if (stats != nullptr && warp_active && i < Tv && (kSW == 4 || half == 0)) {
          // saved for the backward (d2s_attn_policy_bwd): e_ij = 2^(k2 s_ij - m'_i) m_ij, P_ij = e_ij / den_i + c_i
          const float inv = 1.0f / den;
          reinterpret_cast<float4*>(stats)[(size_t)unit * T + i] = make_float4(mxk, inv, c_eps_row * inv, 0.0f);
        }
        if (cls_row != nullptr && t == 0 && warp == 0) {
          // CLS row (query 0 = lane 0 of warp 0): probabilities of row 0, Attention.forward's second output
          __syncwarp();
          const float den0 = __shfl_sync(0xffffffffu, den, 0);
          const float ce0 = __shfl_sync(0xffffffffu, c_eps_row, 0);
          for (int j = lane; j < T; j += 32) cls_row[(size_t)unit * T + j] = (!kVar || j < Tv) ? (cls_s[j] + ce0) / den0 : 0.f;
          __syncwarp();
        }
        // ---- epilogue: this warp's share of the 64 output columns -------------------------------------------
        constexpr int kOC = kSW == 8 ? 32 : 64;            // output columns per warp
        const int oc0 = kSW == 8 ? half * 32 : 0;
        TC_TRACE(6)
        mbar_wait(smem_u32(&bars->o_full), g & 1);
        TC_TRACE(3)
        tc_fence_after();
        if constexpr (kNT == 2) {
          uint32_t ow[kOC / 2];   // packed bf16
          if (warp_active) {
            const float inv = 1.0f / den;
#pragma unroll
            for (int ch = 0; ch < kOC / 16; ++ch) {
              uint32_t v[16];
              tmem_ld16_nowait(lane_addr + (uint32_t)(kOCol + oc0 + ch * 16), v);
              tmem_ld_wait();
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                float o0 = __uint_as_float(v[2 * q]), o1 = __uint_as_float(v[2 * q + 1]);
                if (kPol) {
                  o0 += c_eps_row * vsum_s[oc0 + ch * 16 + 2 * q];
                  o1 += c_eps_row * vsum_s[oc0 + ch * 16 + 2 * q + 1];
                }
                ow[ch * 8 + q] = pack_bf16x2(o0 * inv, o1 * inv);
              }
            }
          }
          // O is in registers: release TMEM so the next tile's S-MMA overlaps the stores
          tc_fence_before();
          mbar_arrive(smem_u32(&bars->tmem_free));
          if (warp_active && i < Tv) {
            uint4* orow = reinterpret_cast<uint4*>(out + ((size_t)b * T + i) * (size_t)(H * kTcHD) + (size_t)h * kTcHD + oc0);
#pragma unroll
            for (int q = 0; q < kOC / 8; ++q) orow[q] = make_uint4(ow[4 * q], ow[4 * q + 1], ow[4 * q + 2], ow[4 * q + 3]);
          }
        } else {
          // 4 CTAs per SM: no registers to spare for the whole row, store chunk by chunk
          if (warp_active) {
            const float inv = 1.0f / den;
            __nv_bfloat16* orow = out + ((size_t)b * T + min(i, Tv - 1)) * (size_t)(H * kTcHD) + (size_t)h * kTcHD;
#pragma unroll
            for (int ch = 0; ch < kTcHD / 16; ++ch) {
              uint32_t v[16];
              tmem_ld16_nowait(lane_addr + (uint32_t)(kOCol + ch * 16), v);
              tmem_ld_wait();
              uint32_t w[8];
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                float o0 = __uint_as_float(v[2 * q]), o1 = __uint_as_float(v[2 * q + 1]);
                if (kPol) {
                  o0 += c_eps_row * vsum_s[ch * 16 + 2 * q];
                  o1 += c_eps_row * vsum_s[ch * 16 + 2 * q + 1];
                }
                w[q] = pack_bf16x2(o0 * inv, o1 * inv);
              }
              if (i < Tv) {
                reinterpret_cast<uint4*>(orow)[ch * 2] = make_uint4(w[0], w[1], w[2], w[3]);
                reinterpret_cast<uint4*>(orow)[ch * 2 + 1] = make_uint4(w[4], w[5], w[6], w[7]);
              }
            }
          }
          tc_fence_before();
          mbar_arrive(smem_u32(&bars->tmem_free));
        }
        if (kVar && i >= Tv && i < T && (kSW == 4 || half == 0)) {   // pad rows of the output: zeros
          uint4* orow = reinterpret_cast<uint4*>(out + ((size_t)b * T + i) * (size_t)(H * kTcHD) + (size_t)h * kTcHD);
#pragma unroll
          for (int q = 0; q < kTcHD / 8; ++q) orow[q] = make_uint4(0u, 0u, 0u, 0u);
        }
        TC_TRACE(4)
      }
    }
    if (warp == 0) { TC_TRACE_DUMP(1) }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kSW) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(kTmemCols) : "memory");
  }
}

// the fp32 attention forward (SIMT kernel, d2s_attn_simt.cu)
int attn_simt_dispatch(const void* qkv, const float* policy, int B, int T, int H, int hd, float scale, float eps, void* out,
                       float* cls_row, cudaStream_t stream, const int* lens = nullptr);

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeFn encode_fn() {
  bind_primary_context();
  static EncodeFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeFn>(p);
  }
  return fn;
}

// 3-D view of the packed qkv buffer: (3*H*64 columns, T tokens, B images); rows past T are zero-filled by TMA.
// map_a: box of min(Tkp,128) rows; map_b: box of the Tkp-128 remaining rows (T > 128 only).
static int encode_qkv_maps(const void* qkv, int B, int T, int H, int Tkp, CUtensorMap& map_a, CUtensorMap& map_b) {
  EncodeFn enc = encode_fn();
  D2S_REQUIRE(enc != nullptr, D2S_ERR_CUDA, "attn_policy_fwd: cuTensorMapEncodeTiled is unavailable from the driver");
  const cuuint64_t gdim[3] = {(cuuint64_t)3 * H * kTcHD, (cuuint64_t)T, (cuuint64_t)B};
  const cuuint64_t gstride[2] = {(cuuint64_t)3 * H * kTcHD * 2, (cuuint64_t)T * 3 * H * kTcHD * 2};
  const cuuint32_t estr[3] = {1, 1, 1};
  const int rows_a = Tkp < kTileRows ? Tkp : kTileRows;
  const int rows_b = Tkp > kTileRows ? Tkp - kTileRows : rows_a;
  for (int m = 0; m < 2; ++m) {
    const cuuint32_t box[3] = {(cuuint32_t)kTcHD, (cuuint32_t)(m == 0 ? rows_a : rows_b), 1};
    CUresult cr = enc(m == 0 ? &map_a : &map_b, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(qkv), gdim, gstride,
                      box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    D2S_REQUIRE(cr == CUDA_SUCCESS, D2S_ERR_CUDA, "attn_policy_fwd: cuTensorMapEncodeTiled failed (%d)", (int)cr);
  }
  return D2S_OK;
}

static size_t tc_smem_bytes(int knt, int Tkp, int kbufs) {
  const int rows_a = knt == 1 ? Tkp : kTileRows, rows_b = knt == 1 ? 0 : Tkp - kTileRows;
  (void)rows_a;
  return 1024 + (size_t)(kTileRows + rows_b) * 128 + (size_t)(kbufs + 1) * Tkp * 128 + sizeof(TcBars) +
         (256 + 256 + 64 + 256 + 256 + 256 + 256) * sizeof(float);
}

template <int kNT, bool kPol, int kSW, bool kVar = false>
static int launch_tc(const CUtensorMap& map_a, const CUtensorMap& map_b, const float* policy, int units, int T, int H,
                     int Tkp, float scale, float eps, void* out, float* cls_row, float* stats, const void* qkv,
                     cudaStream_t stream, const int* lens = nullptr) {
  auto kern = attn_tc_fwd_kernel<kNT, kPol, kSW, kVar>;
  // two K buffers when they still leave room for the intended number of CTAs per SM
  const int per_sm = kNT == 1 ? 4 : 2;
  const size_t budget = (size_t)(228 * 1024) / per_sm - 1024;
  const int kbufs = tc_smem_bytes(kNT, Tkp, 2) <= budget ? 2 : 1;
  const size_t smem = tc_smem_bytes(kNT, Tkp, kbufs);
  static SmemOptIn opt;  // one per instantiation
  cudaError_t e = opt_in_smem(opt, kern, 113 * 1024);
  D2S_REQUIRE(e == cudaSuccess, D2S_ERR_CUDA, "attn_policy_fwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  const int grid = units < per_sm * kNumSMs ? units : per_sm * kNumSMs;
  kern<<<grid, tc_threads(kSW), smem, stream>>>(map_a, map_b, policy, units, T, H, Tkp, kbufs, scale, eps, (__nv_bfloat16*)out,
                                                 cls_row, stats, (const __nv_bfloat16*)qkv, lens);
  count_launch();
  return check_launch(kVar ? "d2s_attn_varlen_fwd(tcgen05)" : "d2s_attn_policy_fwd(tcgen05)");
}

}  // namespace d2s
