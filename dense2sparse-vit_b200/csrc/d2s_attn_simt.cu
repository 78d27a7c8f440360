// Kernel family (4), CUDA-core part:
//   * softmax_with_policy forward/backward over a materialised (B,H,T,T) score tensor -- the drop-in for
//     Attention.softmax_with_policy (vit_models/dynamic_vit.py:195-214) used by the training path, one
//     pass instead of the reference's ~11 elementwise passes;
//   * the fused fp32 attention core (QK^T -> policy softmax -> PV, CLS-row side output) used for the
//     1e-4 fp32 parity runs.  The bf16 production path is the tcgen05 kernel in d2s_attn_tc.cu.
//
//   P_ij = (exp(s_ij - max_j s_ij) * m_ij + eps/T) / (sum_j exp(.) * m_ij + eps),  m_ij = p_j + (1-p_j)[i==j]
#include "d2s_tc.cuh"

namespace d2s {

constexpr int kRowThreads = 256;
constexpr int kRowWarps = kRowThreads / 32;
constexpr int kRowsPerCta = 64;

// bf16 inputs: the reference subtracts the row max in the input dtype before converting to fp32
// (attn - max_att happens before .to(torch.float32), dynamic_vit.py:206-212)
__device__ __forceinline__ float sub_in_dtype(float s, float m, const float*) { return s - m; }
__device__ __forceinline__ float sub_in_dtype(float s, float m, const __nv_bfloat16*) {
  return __bfloat162float(__float2bfloat16_rn(s - m));
}

// One warp per score row; lane owns columns lane + 32*e.  EPL*32 >= T.
template <typename T_, int EPL>
__global__ void __launch_bounds__(kRowThreads)
softmax_policy_fwd_kernel(const T_* __restrict__ attn, const float* __restrict__ policy, int H, int T, float eps,
                          T_* __restrict__ out, float* __restrict__ stats) {
  const int bh = blockIdx.y, b = bh / H;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row_end = min(T, (int)(blockIdx.x + 1) * kRowsPerCta);
  float pol[EPL];
#pragma unroll
  for (int e = 0; e < EPL; ++e) {
    const int j = lane + 32 * e;
    pol[e] = (policy && j < T) ? policy[(size_t)b * T + j] : 1.0f;
  }
  const float c = policy ? eps / (float)T : 0.0f;
  const float eps_den = policy ? eps : 0.0f;
  for (int i = blockIdx.x * kRowsPerCta + warp; i < row_end; i += kRowWarps) {
    const size_t base = ((size_t)bh * T + i) * T;
    float s[EPL];
    float m = -INFINITY;
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      const int j = lane + 32 * e;
      s[e] = (j < T) ? ld_as_float(attn, base + j) : -INFINITY;
      m = fmaxf(m, s[e]);
    }
    m = warp_max(m);
    float sum = 0.f;
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      const int j = lane + 32 * e;
      float a = 0.f;
      if (j < T) {
        const float mask = (j == i) ? 1.0f : pol[e];  // p_j + (1-p_j)*[i==j]
        a = expf(sub_in_dtype(s[e], m, attn)) * mask;
      }
      s[e] = a;
      sum += a;
    }
    sum = warp_sum(sum);
    const float den = sum + eps_den;
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      const int j = lane + 32 * e;
      if (j < T) st_from_float(out, base + j, (s[e] + c) / den);
    }
    if (stats && lane == 0) {
      stats[((size_t)bh * T + i) * 2] = m;
      stats[((size_t)bh * T + i) * 2 + 1] = den;
    }
  }
}

// ---- bf16, padded rows (row stride ld % 8 == 0, T <= 256): lane owns columns 8*lane .. 8*lane+7, one 16-byte access per
// lane and row instead of 2-byte scalars (rows of T = 197 bf16 are only 2-byte aligned when packed densely; the training
// path therefore keeps its score tensors with ld = round_up(T, 8)).  Same arithmetic as the scalar kernels. ----
__device__ __forceinline__ void unpack8(const int4& v, float (&f)[8]) {
  const uint32_t w[4] = {(uint32_t)v.x, (uint32_t)v.y, (uint32_t)v.z, (uint32_t)v.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    f[2 * k] = __uint_as_float(w[k] << 16);
    f[2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u);
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * k], f[2 * k + 1]);
    w[k] = *reinterpret_cast<const uint32_t*>(&h);
  }
  return make_uint4(w[0], w[1], w[2], w[3]);
}

// exp of a non-positive bf16-rounded difference: MUFU.EX2 (relative error 2^-22, far inside bf16)
__device__ __forceinline__ float exp_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
  return y;
}

// Padded-row kernels (rows of `ld` bf16, ld % 8 == 0, the (B*H, rows, ld) head-major score tensor of the training path).
// A CTA owns kRowsPerCta consecutive rows = ONE contiguous block of the tensor, so the whole block is fetched by 1-D bulk
// copies (TMA unit, no tensor map) issued up front by one thread: sub-blocks of one warp step (one or two rows per warp),
// each with its own mbarrier.  Every byte the CTA will read is in flight from the first instruction on (register-staged row loads, even
// with a one-row prefetch, left these kernels latency-bound at 1.2-2.3 TB/s); warps start on sub-block 0 while the rest
// still streams in.  Results go straight to global memory (16 bytes per lane, whole rows per warp).
struct RowBars { unsigned long long full[kRowsPerCta / kRowWarps]; };

// issues the loads of this CTA's row block: `ntens` tensors (1: scores; 2: scores + upstream gradient) side by side in `stage`
template <int kSubRows>
__device__ __forceinline__ void row_block_issue(RowBars* bars, uint8_t* stage, const __nv_bfloat16* t0, const __nv_bfloat16* t1,
                                                size_t block_elem0, int nrows, int ld) {
  const uint32_t row_bytes = (uint32_t)ld * 2u;
  for (int k = 0; k < kRowsPerCta / kSubRows; ++k) {
    const int r0 = k * kSubRows;
    if (r0 >= nrows) break;
    const uint32_t bytes = (uint32_t)min(kSubRows, nrows - r0) * row_bytes;
    const uint32_t bar = smem_u32(&bars->full[k]);
    mbar_expect_tx(bar, t1 ? 2 * bytes : bytes);
    bulk_load_1d(smem_u32(stage + (size_t)r0 * row_bytes), t0 + block_elem0 + (size_t)r0 * ld, bytes, bar);
    if (t1)
      bulk_load_1d(smem_u32(stage + (size_t)(kRowsPerCta + r0) * row_bytes), t1 + block_elem0 + (size_t)r0 * ld, bytes, bar);
  }
}

// Arithmetic is kept to ~10 issue slots per element (the first versions spent ~22 and were ISSUE-bound at 2.4 TB/s whatever
// the load path): the row max and the reference's bf16 `attn - max` are taken on packed bf16x2 words (max.bf16x2 /
// sub.rn.bf16x2), columns >= T are forced to -inf / 0 by two per-lane constant bit masks instead of per-element predicates,
// and the diagonal (m_ii = 1 whatever the policy) is not special-cased per element: rows are computed with m_ij = p_j
// throughout and corrected with the one diagonal element, read as a shared-memory broadcast.
// LPR lanes per row (32, or 16 for ld <= 128: two consecutive rows per warp); lane sl of a row owns columns 8*sl .. 8*sl+7.
__device__ __forceinline__ uint32_t sub_bf16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("sub.rn.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ uint32_t max_bf16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
__device__ __forceinline__ float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
constexpr float kLog2e = 1.4426950408889634f;

template <int LPR>
struct RowMap {
  static constexpr int kRPW = 32 / LPR;                       // rows per warp step
  static constexpr int kSubRows = kRowWarps * kRPW;           // rows per sub-block (one barrier each)
  static constexpr int kSubs = kRowsPerCta / kSubRows;
};

// per-lane constants: keep[w] selects the valid halves of packed word w (columns < T), ninf[w] holds bf16 -inf in the others
__device__ __forceinline__ void lane_masks(int j0, int T, uint32_t (&keep)[4], uint32_t (&ninf)[4]) {
#pragma unroll
  for (int w = 0; w < 4; ++w) {
    keep[w] = (j0 + 2 * w < T ? 0x0000ffffu : 0u) | (j0 + 2 * w + 1 < T ? 0xffff0000u : 0u);
    ninf[w] = ~keep[w] & 0xff80ff80u;
  }
}

template <int LPR>
__global__ void __launch_bounds__(kRowThreads)
softmax_policy_fwd_vec_kernel(const __nv_bfloat16* __restrict__ attn, const float* __restrict__ policy, int H, int T, int rows,
                              int ld, float eps, __nv_bfloat16* __restrict__ out, float* __restrict__ stats) {
  using M = RowMap<LPR>;
  extern __shared__ __align__(128) uint8_t row_stage[];
  __shared__ RowBars bars;
  __shared__ float pol_s[256];
  const int bh = blockIdx.y, b = bh / H;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row0 = blockIdx.x * kRowsPerCta;
  const int row_end = min(T, row0 + kRowsPerCta);
  const size_t block0 = ((size_t)bh * rows + row0) * ld;
  if (threadIdx.x == 0) {
    for (int k = 0; k < M::kSubs; ++k) mbar_init(smem_u32(&bars.full[k]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    row_block_issue<M::kSubRows>(&bars, row_stage, attn, nullptr, block0, row_end - row0, ld);
  }
  for (int j = threadIdx.x; j < 256; j += kRowThreads) pol_s[j] = j < T ? (policy ? policy[(size_t)b * T + j] : 1.0f) : 0.0f;
  const int sl = lane % LPR, sub = lane / LPR;
  const int j0 = sl * 8;
  const bool active = j0 < ld;
  uint32_t keep[4], ninf[4];
  lane_masks(j0, T, keep, ninf);
  const float c = policy ? eps / (float)T : 0.0f;
  const float eps_den = policy ? eps : 0.0f;
  __syncthreads();   // barriers initialised, pol_s filled
  float pol[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) pol[q] = active ? pol_s[j0 + q] : 0.f;
  for (int k = 0; k < M::kSubs; ++k) {
    const int lr = (k * kRowWarps + warp) * M::kRPW;   // first row of this warp step, block-relative
    if (row0 + lr >= row_end) break;
    const int li = lr + sub, i = row0 + li;
    const bool rowok = i < row_end;
    mbar_wait(smem_u32(&bars.full[k]), 0);
    const uint8_t* srow = row_stage + (size_t)(rowok ? li : lr) * ld * 2;
    int4 raw = make_int4(0, 0, 0, 0);
    if (active) raw = *reinterpret_cast<const int4*>(srow + j0 * 2);
    uint32_t w[4] = {(uint32_t)raw.x, (uint32_t)raw.y, (uint32_t)raw.z, (uint32_t)raw.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) w[q] = (w[q] & keep[q]) | ninf[q];
    uint32_t m2 = max_bf16x2(max_bf16x2(w[0], w[1]), max_bf16x2(w[2], w[3]));
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) m2 = max_bf16x2(m2, __shfl_xor_sync(0xffffffffu, m2, o));
    const float m = fmaxf(__uint_as_float(m2 << 16), __uint_as_float(m2 & 0xffff0000u));
    const uint32_t mb = __float_as_uint(m) >> 16;   // m is a bf16 value
    const uint32_t mm = mb | (mb << 16);
    // element pairs on the packed fp32x2 pipe (the kernel is close to issue-bound)
    uint64_t a2[4];
    uint64_t sum2 = f2_bcast(0.f);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t d = sub_bf16x2(w[q], mm);
      float x0, x1;
      f2_unpack(f2_mul(f2_pack(__uint_as_float(d << 16), __uint_as_float(d & 0xffff0000u)), f2_bcast(kLog2e)), x0, x1);
      a2[q] = f2_mul(f2_pack(ex2_fast(x0), ex2_fast(x1)), f2_pack(pol[2 * q], pol[2 * q + 1]));
      sum2 = f2_add(sum2, a2[q]);
    }
    float sum, sum_hi;
    f2_unpack(sum2, sum, sum_hi);
    sum += sum_hi;
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    // diagonal: the reference's mask is 1 there
    const int id = rowok ? i : row0 + lr;
    const float sd = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(srow)[id]);
    const float exd = ex2_fast(__bfloat162float(__float2bfloat16_rn(sd - m)) * kLog2e);
    sum += exd * (1.0f - pol_s[id]);
    const float den = sum + eps_den;
    const float rden = 1.0f / den;
    const float crden = c * rden;
    if (active && rowok) {
      uint32_t pk[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {   // padding columns are written as zeros
        float p0, p1;
        f2_unpack(f2_fma(a2[q], f2_bcast(rden), f2_bcast(crden)), p0, p1);
        pk[q] = pack_bf16x2(p0, p1) & keep[q];
      }
      __nv_bfloat16* orow = out + block0 + (size_t)li * ld;
      *reinterpret_cast<uint4*>(orow + j0) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
      if (sl == (i >> 3)) orow[i] = __float2bfloat16_rn((exd + c) * rden);   // same thread as the vector store: ordered
      if (stats && sl == 0) *reinterpret_cast<float2*>(stats + ((size_t)bh * T + i) * 2) = make_float2(m, den);
    }
  }
  // padding rows T..rows-1 of `out` (the padded tensor is a GEMM operand)
  if (blockIdx.x == gridDim.x - 1 && lane * 8 < ld)
    for (int i = T + warp; i < rows; i += kRowWarps)
      *reinterpret_cast<uint4*>(out + ((size_t)bh * rows + i) * ld + lane * 8) = make_uint4(0, 0, 0, 0);
}

// The gradient through the subtracted row max (dense kernel above: routed to the first argmax) is sum_j dS_ij = O(eps) * g,
// i.e. 1e-6 relative: below bf16 resolution, so this bf16-only kernel leaves it out (and with it the argmax bookkeeping).
template <int LPR>
__global__ void __launch_bounds__(kRowThreads, 3)
softmax_policy_bwd_vec_kernel(const __nv_bfloat16* __restrict__ attn, const float* __restrict__ policy,
                              const __nv_bfloat16* __restrict__ gout, const float* __restrict__ stats, int H, int T, int rows,
                              int ld, float eps, __nv_bfloat16* __restrict__ gattn, float* __restrict__ gpolicy) {
  using M = RowMap<LPR>;
  extern __shared__ __align__(128) uint8_t row_stage[];   // scores block, then gradient block
  __shared__ RowBars bars;
  __shared__ float pol_s[256];
  __shared__ float gp_fix[kRowsPerCta];                   // d policy_i the row loop over-counts on the diagonal
  __shared__ float gp_s[kRowWarps * M::kRPW][LPR * 8];    // per-(warp, row slot) partial d policy (no shared float atomics: CAS loops)
  const int bh = blockIdx.y, b = bh / H;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row0 = blockIdx.x * kRowsPerCta;
  const int row_end = min(T, row0 + kRowsPerCta);
  const size_t block0 = ((size_t)bh * rows + row0) * ld;
  if (threadIdx.x == 0) {
    for (int k = 0; k < M::kSubs; ++k) mbar_init(smem_u32(&bars.full[k]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    row_block_issue<M::kSubRows>(&bars, row_stage, attn, gout, block0, row_end - row0, ld);
  }
  for (int j = threadIdx.x; j < 256; j += kRowThreads) pol_s[j] = j < T ? (policy ? policy[(size_t)b * T + j] : 1.0f) : 0.0f;
  if (threadIdx.x < kRowsPerCta) gp_fix[threadIdx.x] = 0.f;
  const int sl = lane % LPR, sub = lane / LPR;
  const int j0 = sl * 8;
  const bool active = j0 < ld;
  const bool want_gp = gpolicy && policy;
  uint32_t keep[4], ninf[4];
  lane_masks(j0, T, keep, ninf);
  const float c = policy ? eps / (float)T : 0.0f;
  // (max, denominator) of this warp's rows: lane k*kRPW + s holds the pair of warp step k, row slot s
  float2 st = make_float2(0.f, 1.f);
  {
    const int i = row0 + ((lane / M::kRPW) * kRowWarps + warp) * M::kRPW + lane % M::kRPW;
    if (lane < M::kSubs * M::kRPW && i < row_end) st = *reinterpret_cast<const float2*>(stats + ((size_t)bh * T + i) * 2);
  }
  const uint8_t* g_stage = row_stage + (size_t)kRowsPerCta * ld * 2;
  __syncthreads();   // barriers initialised, pol_s filled
  float pol[8];
  uint64_t gp2[4];
#pragma unroll
  for (int q = 0; q < 8; ++q) pol[q] = active ? pol_s[j0 + q] : 0.f;
#pragma unroll
  for (int q = 0; q < 4; ++q) gp2[q] = f2_bcast(0.f);
  for (int k = 0; k < M::kSubs; ++k) {
    const int lr = (k * kRowWarps + warp) * M::kRPW;
    if (row0 + lr >= row_end) break;
    const int li = lr + sub, i = row0 + li;
    const bool rowok = i < row_end;
    const float m = __shfl_sync(0xffffffffu, st.x, k * M::kRPW + sub);
    const float den = __shfl_sync(0xffffffffu, st.y, k * M::kRPW + sub);
    const float rden = rowok ? 1.0f / den : 0.0f;   // a missing second row (last warp step of a block) contributes nothing
    mbar_wait(smem_u32(&bars.full[k]), 0);
    const size_t roff = (size_t)(rowok ? li : lr) * ld * 2;
    int4 sraw = make_int4(0, 0, 0, 0), graw = sraw;
    if (active) {
      sraw = *reinterpret_cast<const int4*>(row_stage + roff + j0 * 2);
      graw = *reinterpret_cast<const int4*>(g_stage + roff + j0 * 2);
    }
    const uint32_t sw[4] = {(uint32_t)sraw.x, (uint32_t)sraw.y, (uint32_t)sraw.z, (uint32_t)sraw.w};
    const uint32_t gw[4] = {(uint32_t)graw.x, (uint32_t)graw.y, (uint32_t)graw.z, (uint32_t)graw.w};
    const uint32_t mb = __float_as_uint(m) >> 16;   // the forward's row max is a bf16 value
    const uint32_t mm = mb | (mb << 16);
    // element pairs on the packed fp32x2 pipe (the kernel is close to issue-bound)
    uint64_t g2[4], ex2v[4], a2[4];
    uint64_t part2 = f2_bcast(0.f), gsum2 = f2_bcast(0.f);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t d = sub_bf16x2((sw[q] & keep[q]) | ninf[q], mm);
      const uint32_t gq = gw[q] & keep[q];
      float x0, x1;
      f2_unpack(f2_mul(f2_pack(__uint_as_float(d << 16), __uint_as_float(d & 0xffff0000u)), f2_bcast(kLog2e)), x0, x1);
      ex2v[q] = f2_pack(ex2_fast(x0), ex2_fast(x1));
      g2[q] = f2_pack(__uint_as_float(gq << 16), __uint_as_float(gq & 0xffff0000u));
      a2[q] = f2_mul(ex2v[q], f2_pack(pol[2 * q], pol[2 * q + 1]));
      part2 = f2_fma(g2[q], a2[q], part2);
      gsum2 = f2_add(gsum2, g2[q]);
    }
    float part, part_hi;
    f2_unpack(f2_fma(f2_bcast(c), gsum2, part2), part, part_hi);
    part += part_hi;
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    // diagonal element (mask 1 in the reference, p_i in the sums above)
    const int id = rowok ? i : row0 + lr;
    const float sd = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(row_stage + roff)[id]);
    const float gd = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(g_stage + roff)[id]);
    const float exd = ex2_fast(__bfloat162float(__float2bfloat16_rn(sd - m)) * kLog2e);
    const float gdr = (part + gd * exd * (1.0f - pol_s[id])) * rden * rden;   // (g . P) / den
    uint32_t dsw[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint64_t da = f2_fma(g2[q], f2_bcast(rden), f2_bcast(-gdr));
      float d0, d1;
      f2_unpack(f2_mul(da, a2[q]), d0, d1);       // a == 0 outside the row
      dsw[q] = pack_bf16x2(d0, d1);
      gp2[q] = f2_fma(da, ex2v[q], gp2[q]);       // includes the diagonal: taken out again through gp_fix
    }
    if (active && rowok) {
      __nv_bfloat16* drow = gattn + block0 + (size_t)li * ld;
      *reinterpret_cast<uint4*>(drow + j0) = make_uint4(dsw[0], dsw[1], dsw[2], dsw[3]);
      const float dsd = fmaf(gd, rden, -gdr) * exd;
      if (sl == (i >> 3)) drow[i] = __float2bfloat16_rn(dsd);   // same thread as the vector store: ordered
      if (sl == 0) gp_fix[li] = dsd;
    }
  }
  if (want_gp) {
    float* mine = gp_s[warp * M::kRPW + sub];
    float gp[8];
#pragma unroll
    for (int q = 0; q < 4; ++q) f2_unpack(gp2[q], gp[2 * q], gp[2 * q + 1]);
    *reinterpret_cast<float4*>(mine + j0) = make_float4(gp[0], gp[1], gp[2], gp[3]);
    *reinterpret_cast<float4*>(mine + j0 + 4) = make_float4(gp[4], gp[5], gp[6], gp[7]);
    __syncthreads();
    for (int j = threadIdx.x; j < T; j += kRowThreads) {
      float acc = 0.f;
#pragma unroll
      for (int w = 0; w < kRowWarps * M::kRPW; ++w) acc += gp_s[w][j];
      if (j >= row0 && j < row_end) acc -= gp_fix[j - row0];
      atomicAdd(&gpolicy[(size_t)b * T + j], acc);
    }
  }
}

template <typename T_, int EPL>
__global__ void __launch_bounds__(kRowThreads)
softmax_policy_bwd_kernel(const T_* __restrict__ attn, const float* __restrict__ policy, const T_* __restrict__ gout,
                          const float* __restrict__ stats, int H, int T, float eps, T_* __restrict__ gattn,
                          float* __restrict__ gpolicy) {
  __shared__ float gp_s[EPL * 32];
  const int bh = blockIdx.y, b = bh / H;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row_end = min(T, (int)(blockIdx.x + 1) * kRowsPerCta);
  for (int j = threadIdx.x; j < EPL * 32; j += kRowThreads) gp_s[j] = 0.f;
  __syncthreads();
  float pol[EPL], gp[EPL];
#pragma unroll
  for (int e = 0; e < EPL; ++e) {
    const int j = lane + 32 * e;
    pol[e] = (policy && j < T) ? policy[(size_t)b * T + j] : 1.0f;
    gp[e] = 0.f;
  }
  const float c = policy ? eps / (float)T : 0.0f;
  for (int i = blockIdx.x * kRowsPerCta + warp; i < row_end; i += kRowWarps) {
    const size_t base = ((size_t)bh * T + i) * T;
    const float m = stats[((size_t)bh * T + i) * 2];
    const float den = stats[((size_t)bh * T + i) * 2 + 1];
    float ex[EPL], a[EPL], g[EPL];
    float gdotp = 0.f;
    // first-occurrence argmax of the row (torch.max backward routes the max-term there)
    float best = -INFINITY;
    int best_j = 0x7fffffff;
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      const int j = lane + 32 * e;
      ex[e] = a[e] = g[e] = 0.f;
      if (j < T) {
        const float s = ld_as_float(attn, base + j);
        if (s > best) { best = s; best_j = j; }
        const float mask = (j == i) ? 1.0f : pol[e];
        ex[e] = expf(sub_in_dtype(s, m, attn));
        a[e] = ex[e] * mask;
        g[e] = ld_as_float(gout, base + j);
        gdotp += g[e] * ((a[e] + c) / den);
      }
    }
    gdotp = warp_sum(gdotp);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oj = __shfl_xor_sync(0xffffffffu, best_j, o);
      if (ob > best || (ob == best && oj < best_j)) { best = ob; best_j = oj; }
    }
    float ds[EPL];
    float ds_sum = 0.f;
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      const int j = lane + 32 * e;
      const float da = (g[e] - gdotp) / den;  // dL/da_ij
      ds[e] = da * a[e];
      ds_sum += ds[e];
      if (j < T && j != i) gp[e] += da * ex[e];  // dL/dp_j, diagonal excluded (m_ii == 1)
    }
    ds_sum = policy ? warp_sum(ds_sum) : 0.f;  // plain softmax: the max-term vanishes identically
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      const int j = lane + 32 * e;
      if (j < T) st_from_float(gattn, base + j, ds[e] - (j == best_j ? ds_sum : 0.f));
    }
  }
  if (gpolicy && policy) {
#pragma unroll
    for (int e = 0; e < EPL; ++e) atomicAdd(&gp_s[lane + 32 * e], gp[e]);
    __syncthreads();
    for (int j = threadIdx.x; j < T; j += kRowThreads) atomicAdd(&gpolicy[(size_t)b * T + j], gp_s[j]);
  }
}

// ---------------------------------------------------------------------------------------------------
// Fused fp32 attention core.  CTA = (row chunk, b*H + h): K and V of the head staged in shared memory
// as fp32 (K rows padded to HD+1 floats so lane-per-key reads are bank-conflict free); each warp
// processes kQR query rows per pass: scores (lane owns keys lane+32e), policy softmax, then PV with
// lane owning output dims lane and lane+32.
constexpr int kAttnThreads = 256;
constexpr int kAttnWarps = kAttnThreads / 32;
constexpr int kQR = 4;       // query rows per warp pass
constexpr int kAttnEPL = 8;  // T <= 256

// kVar: variable-length form (d2s_attn_varlen_fwd): image b has Tv = lens[b] valid tokens of its T (padded) rows; rows and cls_row
// columns Tv..T-1 are written as zeros (no policy)
template <typename T_, int HD, bool kVar = false>
__global__ void __launch_bounds__(kAttnThreads)
attn_simt_fwd_kernel(const T_* __restrict__ qkv, const float* __restrict__ policy, int T, int H, float scale, float eps,
                     T_* __restrict__ out, float* __restrict__ cls_row, int rows_per_cta, const int* __restrict__ lens) {
  extern __shared__ float sm[];
  float* Ks = sm;                                  // T x (HD+1)
  float* Vs = Ks + (size_t)T * (HD + 1);           // T x HD
  float* pol_s = Vs + (size_t)T * HD;              // T
  float* qs = pol_s + ((T + 3) & ~3);              // warps x kQR x HD
  float* ps = qs + kAttnWarps * kQR * HD;          // warps x kQR x T
  const int bh = blockIdx.y, b = bh / H, h = bh % H;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t tok_stride = (size_t)3 * H * HD;
  const T_* q_base = qkv + (size_t)b * T * tok_stride + (size_t)h * HD;
  const T_* k_base = q_base + (size_t)H * HD;
  const T_* v_base = q_base + (size_t)2 * H * HD;
  const int Tv = kVar ? min(max(lens[b], 0), T) : T;
  for (int idx = threadIdx.x; idx < Tv * HD; idx += kAttnThreads) {
    const int j = idx / HD, d = idx % HD;
    Ks[j * (HD + 1) + d] = ld_as_float(k_base, (size_t)j * tok_stride + d);
    Vs[j * HD + d] = ld_as_float(v_base, (size_t)j * tok_stride + d);
  }
  for (int j = threadIdx.x; j < T; j += kAttnThreads) pol_s[j] = policy ? policy[(size_t)b * T + j] : 1.0f;
  __syncthreads();
  const float c = policy ? eps / (float)T : 0.0f;
  const float eps_den = policy ? eps : 0.0f;
  float* my_q = qs + warp * kQR * HD;
  float* my_p = ps + (size_t)warp * kQR * T;
  const int row_begin = blockIdx.x * rows_per_cta;
  const int row_end = min(Tv, row_begin + rows_per_cta);
  if (kVar) {   // pad rows of this CTA's row range and the CLS row's pad columns: zeros
    for (int idx = threadIdx.x; idx < (min(T, row_begin + rows_per_cta) - max(row_begin, Tv)) * HD; idx += kAttnThreads)
      st_from_float(out, ((size_t)b * T + max(row_begin, Tv) + idx / HD) * (size_t)(H * HD) + (size_t)h * HD + idx % HD, 0.f);
    if (cls_row && blockIdx.x == 0)
      for (int j = Tv + threadIdx.x; j < T; j += kAttnThreads) cls_row[(size_t)bh * T + j] = 0.f;
  }
  for (int i0 = row_begin + warp * kQR; i0 < row_end; i0 += kAttnWarps * kQR) {
#pragma unroll
    for (int r = 0; r < kQR; ++r) {
      const int i = min(i0 + r, Tv - 1);
      for (int d = lane; d < HD; d += 32) my_q[r * HD + d] = ld_as_float(q_base, (size_t)i * tok_stride + d) * scale;
    }
    __syncwarp();
    float s[kQR][kAttnEPL];
#pragma unroll
    for (int r = 0; r < kQR; ++r)
#pragma unroll
      for (int e = 0; e < kAttnEPL; ++e) s[r][e] = 0.f;
    for (int d = 0; d < HD; ++d) {
      float qd[kQR];
#pragma unroll
      for (int r = 0; r < kQR; ++r) qd[r] = my_q[r * HD + d];
#pragma unroll
      for (int e = 0; e < kAttnEPL; ++e) {
        const int j = lane + 32 * e;
        if (j < Tv) {
          const float kv = Ks[j * (HD + 1) + d];
#pragma unroll
          for (int r = 0; r < kQR; ++r) s[r][e] = fmaf(qd[r], kv, s[r][e]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < kQR; ++r) {
      const int i = i0 + r;
      float m = -INFINITY;
#pragma unroll
      for (int e = 0; e < kAttnEPL; ++e) if (lane + 32 * e < Tv) m = fmaxf(m, s[r][e]);
      m = warp_max(m);
      float sum = 0.f;
#pragma unroll
      for (int e = 0; e < kAttnEPL; ++e) {
        const int j = lane + 32 * e;
        float a = 0.f;
        if (j < Tv) a = expf(s[r][e] - m) * ((j == i) ? 1.0f : pol_s[j]);
        s[r][e] = a;
        sum += a;
      }
      sum = warp_sum(sum);
      const float den = sum + eps_den;
#pragma unroll
      for (int e = 0; e < kAttnEPL; ++e) {
        const int j = lane + 32 * e;
        if (j < Tv) {
          const float p = (s[r][e] + c) / den;
          my_p[r * T + j] = p;
          if (cls_row && i == 0) cls_row[(size_t)bh * T + j] = p;
        }
      }
    }
    __syncwarp();
    float o[kQR][HD / 32];
#pragma unroll
    for (int r = 0; r < kQR; ++r)
#pragma unroll
      for (int q = 0; q < HD / 32; ++q) o[r][q] = 0.f;
    for (int j = 0; j < Tv; ++j) {
      float vv[HD / 32];
#pragma unroll
      for (int q = 0; q < HD / 32; ++q) vv[q] = Vs[j * HD + lane + 32 * q];
#pragma unroll
      for (int r = 0; r < kQR; ++r) {
        const float p = my_p[r * T + j];
#pragma unroll
        for (int q = 0; q < HD / 32; ++q) o[r][q] = fmaf(p, vv[q], o[r][q]);
      }
    }
#pragma unroll
    for (int r = 0; r < kQR; ++r) {
      const int i = i0 + r;
      if (i < row_end) {
#pragma unroll
        for (int q = 0; q < HD / 32; ++q)
          st_from_float(out, ((size_t)b * T + i) * (size_t)(H * HD) + (size_t)h * HD + lane + 32 * q, o[r][q]);
      }
    }
    __syncwarp();
  }
}

template <typename T_, int HD>
static int launch_attn_simt(const void* qkv, const float* policy, int B, int T, int H, float scale, float eps, void* out,
                            float* cls_row, cudaStream_t stream, const int* lens) {
  const size_t smem = sizeof(float) * ((size_t)T * (HD + 1) + (size_t)T * HD + ((T + 3) & ~3) +
                                       (size_t)kAttnWarps * kQR * HD + (size_t)kAttnWarps * kQR * T);
  D2S_REQUIRE(smem <= 227 * 1024, D2S_ERR_ARG, "attn(simt): T=%d needs %zu B of shared memory", T, smem);
  auto kern = lens ? attn_simt_fwd_kernel<T_, HD, true> : attn_simt_fwd_kernel<T_, HD>;
  static SmemOptIn opt[2];  // one per kernel instantiation
  cudaError_t e = opt_in_smem(opt[lens ? 1 : 0], kern, 227 * 1024);
  D2S_REQUIRE(e == cudaSuccess, D2S_ERR_CUDA, "attn(simt): cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  // enough CTAs to fill the machine: split the query rows when B*H is small
  int chunks = ceil_div(2 * kNumSMs, B * H);
  const int max_chunks = ceil_div(T, kAttnWarps * kQR);
  chunks = chunks < 1 ? 1 : (chunks > max_chunks ? max_chunks : chunks);
  const int rows_per_cta = ceil_div(ceil_div(T, chunks), kQR) * kQR;
  dim3 grid(ceil_div(T, rows_per_cta), B * H);
  kern<<<grid, kAttnThreads, smem, stream>>>((const T_*)qkv, policy, T, H, scale, eps, (T_*)out, cls_row, rows_per_cta, lens);
  count_launch();
  return check_launch(lens ? "d2s_attn_varlen_fwd(simt)" : "d2s_attn_policy_fwd(simt)");
}

int attn_simt_dispatch(const void* qkv, const float* policy, int B, int T, int H, int hd, float scale, float eps, void* out,
                       float* cls_row, cudaStream_t stream, const int* lens) {
  D2S_REQUIRE(hd == 64 || hd == 32, D2S_ERR_ARG, "attn(simt): hd=%d unsupported (32 or 64)", hd);
  D2S_REQUIRE(T >= 1 && T <= 32 * kAttnEPL, D2S_ERR_ARG, "attn(simt): T=%d outside [1,%d]", T, 32 * kAttnEPL);
  return hd == 64 ? launch_attn_simt<float, 64>(qkv, policy, B, T, H, scale, eps, out, cls_row, stream, lens)
                  : launch_attn_simt<float, 32>(qkv, policy, B, T, H, scale, eps, out, cls_row, stream, lens);
}

}  // namespace d2s

using namespace d2s;

template <typename T_>
static int launch_swp_fwd(const void* attn, const float* policy, int B, int H, int T, float eps, void* out, float* stats,
                          cudaStream_t stream) {
  dim3 grid(ceil_div(T, kRowsPerCta), B * H);
  if (T <= 256)
    softmax_policy_fwd_kernel<T_, 8><<<grid, kRowThreads, 0, stream>>>((const T_*)attn, policy, H, T, eps, (T_*)out, stats);
  else
    softmax_policy_fwd_kernel<T_, 32><<<grid, kRowThreads, 0, stream>>>((const T_*)attn, policy, H, T, eps, (T_*)out, stats);
  count_launch();
  return check_launch("d2s_softmax_policy_fwd");
}

template <typename T_>
static int launch_swp_bwd(const void* attn, const float* policy, const void* gout, const float* stats, int B, int H, int T,
                          float eps, void* gattn, float* gpolicy, cudaStream_t stream) {
  dim3 grid(ceil_div(T, kRowsPerCta), B * H);
  if (T <= 256)
    softmax_policy_bwd_kernel<T_, 8><<<grid, kRowThreads, 0, stream>>>((const T_*)attn, policy, (const T_*)gout, stats, H, T,
                                                                      eps, (T_*)gattn, gpolicy);
  else
    softmax_policy_bwd_kernel<T_, 32><<<grid, kRowThreads, 0, stream>>>((const T_*)attn, policy, (const T_*)gout, stats, H, T,
                                                                       eps, (T_*)gattn, gpolicy);
  count_launch();
  return check_launch("d2s_softmax_policy_bwd");
}

extern "C" int d2s_softmax_policy_fwd(const void* attn, const float* policy, int dtype, int B, int H, int T, float eps,
                                      void* out, float* stats, d2s_stream_t stream) {
  D2S_REQUIRE(attn && out, D2S_ERR_ARG, "softmax_policy_fwd: null pointer");
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "softmax_policy_fwd: dtype %d unsupported", dtype);
  D2S_REQUIRE(B >= 0 && H >= 1 && T >= 1 && T <= 1024, D2S_ERR_ARG, "softmax_policy_fwd: bad shape B=%d H=%d T=%d", B, H, T);
  D2S_REQUIRE((long long)B * H <= 65535, D2S_ERR_ARG, "softmax_policy_fwd: B*H=%lld exceeds 65535", (long long)B * H);
  if (B == 0) return D2S_OK;
  return dtype == D2S_F32 ? launch_swp_fwd<float>(attn, policy, B, H, T, eps, out, stats, (cudaStream_t)stream)
                          : launch_swp_fwd<__nv_bfloat16>(attn, policy, B, H, T, eps, out, stats, (cudaStream_t)stream);
}

extern "C" int d2s_softmax_policy_bwd(const void* attn, const float* policy, const void* gout, const float* stats, int dtype,
                                      int B, int H, int T, float eps, void* gattn, float* gpolicy, d2s_stream_t stream) {
  D2S_REQUIRE(attn && gout && stats && gattn, D2S_ERR_ARG, "softmax_policy_bwd: null pointer");
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "softmax_policy_bwd: dtype %d unsupported", dtype);
  D2S_REQUIRE(B >= 0 && H >= 1 && T >= 1 && T <= 1024, D2S_ERR_ARG, "softmax_policy_bwd: bad shape B=%d H=%d T=%d", B, H, T);
  D2S_REQUIRE((long long)B * H <= 65535, D2S_ERR_ARG, "softmax_policy_bwd: B*H=%lld exceeds 65535", (long long)B * H);
  if (B == 0) return D2S_OK;
  return dtype == D2S_F32
             ? launch_swp_bwd<float>(attn, policy, gout, stats, B, H, T, eps, gattn, gpolicy, (cudaStream_t)stream)
             : launch_swp_bwd<__nv_bfloat16>(attn, policy, gout, stats, B, H, T, eps, gattn, gpolicy, (cudaStream_t)stream);
}

/* Padded-row variants for the training attention (bf16, row stride ld % 8 == 0, ld >= T, T <= 256): attn / out / gout / gattn
 * are (B,H,T,ld); out may not alias attn, gattn may alias gout. */
extern "C" int d2s_softmax_policy_fwd_ld(const void* attn, const float* policy, int B, int H, int T, int rows, int ld, float eps,
                                         void* out, float* stats, d2s_stream_t stream) {
  D2S_REQUIRE(attn && out, D2S_ERR_ARG, "softmax_policy_fwd_ld: null pointer");
  D2S_REQUIRE(B >= 0 && H >= 1 && T >= 1 && T <= 256 && rows >= T && ld >= T && ld % 8 == 0 && ld <= 256, D2S_ERR_ARG,
              "softmax_policy_fwd_ld: bad shape B=%d H=%d T=%d rows=%d ld=%d (need T <= rows, T <= ld <= 256, ld %% 8 == 0)", B, H, T,
              rows, ld);
  D2S_REQUIRE((long long)B * H <= 65535, D2S_ERR_ARG, "softmax_policy_fwd_ld: B*H=%lld exceeds 65535", (long long)B * H);
  D2S_REQUIRE(aligned16(attn) && aligned16(out), D2S_ERR_ALIGN, "softmax_policy_fwd_ld: pointers must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  dim3 grid(ceil_div(T, kRowsPerCta), B * H);
  const size_t smem = (size_t)kRowsPerCta * ld * 2;
  if (ld <= 128)
    softmax_policy_fwd_vec_kernel<16><<<grid, kRowThreads, smem, (cudaStream_t)stream>>>((const __nv_bfloat16*)attn, policy, H, T,
                                                                                        rows, ld, eps, (__nv_bfloat16*)out, stats);
  else
    softmax_policy_fwd_vec_kernel<32><<<grid, kRowThreads, smem, (cudaStream_t)stream>>>((const __nv_bfloat16*)attn, policy, H, T,
                                                                                        rows, ld, eps, (__nv_bfloat16*)out, stats);
  count_launch();
  return check_launch("d2s_softmax_policy_fwd_ld");
}

extern "C" int d2s_softmax_policy_bwd_ld(const void* attn, const float* policy, const void* gout, const float* stats, int B, int H,
                                         int T, int rows, int ld, float eps, void* gattn, float* gpolicy, d2s_stream_t stream) {
  D2S_REQUIRE(attn && gout && stats && gattn, D2S_ERR_ARG, "softmax_policy_bwd_ld: null pointer");
  D2S_REQUIRE(B >= 0 && H >= 1 && T >= 1 && T <= 256 && rows >= T && ld >= T && ld % 8 == 0 && ld <= 256, D2S_ERR_ARG,
              "softmax_policy_bwd_ld: bad shape B=%d H=%d T=%d rows=%d ld=%d (need T <= rows, T <= ld <= 256, ld %% 8 == 0)", B, H, T,
              rows, ld);
  D2S_REQUIRE((long long)B * H <= 65535, D2S_ERR_ARG, "softmax_policy_bwd_ld: B*H=%lld exceeds 65535", (long long)B * H);
  D2S_REQUIRE(aligned16(attn) && aligned16(gout) && aligned16(gattn), D2S_ERR_ALIGN,
              "softmax_policy_bwd_ld: pointers must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  dim3 grid(ceil_div(T, kRowsPerCta), B * H);
  const size_t smem = (size_t)2 * kRowsPerCta * ld * 2;   // scores block + gradient block (<= 64 KB at ld = 256)
  static SmemOptIn opt;
  cudaError_t e = opt_in_smem(opt, softmax_policy_bwd_vec_kernel<32>, 64 * 1024);
  D2S_REQUIRE(e == cudaSuccess, D2S_ERR_CUDA, "softmax_policy_bwd_ld: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  if (ld <= 128)
    softmax_policy_bwd_vec_kernel<16><<<grid, kRowThreads, smem, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)attn, policy, (const __nv_bfloat16*)gout, stats, H, T, rows, ld, eps, (__nv_bfloat16*)gattn, gpolicy);
  else
    softmax_policy_bwd_vec_kernel<32><<<grid, kRowThreads, smem, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)attn, policy, (const __nv_bfloat16*)gout, stats, H, T, rows, ld, eps, (__nv_bfloat16*)gattn, gpolicy);
  count_launch();
  return check_launch("d2s_softmax_policy_bwd_ld");
}
