// Kernel family (1): stable top-K selection over the N (<=1024, 196 in practice) token scores of an
// image, the fused predictor tails that produce those scores, and the Gumbel keep decision.
//
// One CTA per image.  Scores are mapped to order-preserving 32-bit keys in shared memory and every
// token computes its stable descending rank by counting (N*N/256 compares per thread; 196 tokens ->
// ~150 iterations of LDS-broadcast + compare).  Rank < K decides "kept"; for the ascending-index
// output the position is a ballot/popc prefix.  This is exact (integer) work: bit-exact against
// torch.sort(stable=True, descending=True).
//
// Standalone select moves 4N + 8N bytes per image (2.3 KB): it is launch/latency bound, not HBM bound
// (SURVEY.md section 7 hard part 7); the fused tails read the (N, C) hidden activations (e*N*C bytes) as well.
#include "d2s_tc.cuh"

namespace d2s {

constexpr int kSelThreads = 256;
constexpr int kSelWarps = kSelThreads / 32;
constexpr int kSelMaxN = 1024;
constexpr int kSelEPT = kSelMaxN / kSelThreads;  // elements per thread

struct SelSmem {
  alignas(16) uint32_t key[kSelMaxN + 4];
  int warp_cnt[kSelEPT][kSelWarps];
  float red[kSelWarps];
  float bcast;
};

// All threads of the CTA call this after s.key[0..N) is filled and __syncthreads() has been issued.
__device__ void block_select_write(SelSmem& s, int N, int K, int order, int64_t* __restrict__ kept_b,
                                   int64_t* __restrict__ dropped_b, const float* __restrict__ prev_b = nullptr,
                                   float* __restrict__ prev_kept_b = nullptr) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t mykey[kSelEPT];
  int rank[kSelEPT];
#pragma unroll
  for (int e = 0; e < kSelEPT; ++e) {
    const int i = e * kSelThreads + tid;
    mykey[e] = (i < N) ? s.key[i] : 0u;
    rank[e] = 0;
  }
  const int nchunks = (N + kSelThreads - 1) / kSelThreads;
  if (nchunks == 1) {
    // N <= 256 (196 / 137 / 96 in the models): four keys per 16-byte broadcast load, loop unrolled so that several
    // loads are in flight.  The caller pads s.key[N .. round_up(N,4)) with 0, which is below every real key
    // (float_to_ordered never returns 0), so padded entries never count.
    const uint4* k4 = reinterpret_cast<const uint4*>(s.key);
    const uint32_t my = mykey[0];
    const int i = tid;
    int r0 = 0, r1 = 0, r2 = 0, r3 = 0;
    const int n4 = (N + 3) >> 2;
#pragma unroll 8
    for (int j4 = 0; j4 < n4; ++j4) {
      const uint4 k = k4[j4];
      const int j = 4 * j4;
      r0 += (k.x > my) || (k.x == my && j < i);
      r1 += (k.y > my) || (k.y == my && j + 1 < i);
      r2 += (k.z > my) || (k.z == my && j + 2 < i);
      r3 += (k.w > my) || (k.w == my && j + 3 < i);
    }
    rank[0] = (r0 + r1) + (r2 + r3);
  } else {
    for (int j = 0; j < N; ++j) {
      const uint32_t kj = s.key[j];  // broadcast read
#pragma unroll
      for (int e = 0; e < kSelEPT; ++e) {
        if (e < nchunks) {
          const int i = e * kSelThreads + tid;
          rank[e] += (kj > mykey[e]) || (kj == mykey[e] && j < i);
        }
      }
    }
  }
  if (order == D2S_ORDER_SCORE_DESC) {
#pragma unroll
    for (int e = 0; e < kSelEPT; ++e) {
      const int i = e * kSelThreads + tid;
      if (i < N) {
        if (rank[e] < K) {
          if (kept_b) kept_b[rank[e]] = i;
          if (prev_kept_b) prev_kept_b[rank[e]] = prev_b ? prev_b[i] : 1.0f;  // batch_index_select(prev_decision, keep)
        } else if (dropped_b) dropped_b[rank[e] - K] = i;
      }
    }
    return;
  }
  // ascending-index output: position = number of kept tokens with a smaller index
  unsigned ball[kSelEPT];
#pragma unroll
  for (int e = 0; e < kSelEPT; ++e) {
    const int i = e * kSelThreads + tid;
    const bool keep = (i < N) && (rank[e] < K);
    ball[e] = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) s.warp_cnt[e][warp] = __popc(ball[e]);
  }
  __syncthreads();
#pragma unroll
  for (int e = 0; e < kSelEPT; ++e) {
    const int i = e * kSelThreads + tid;
    if (i >= N) continue;
    int before = 0;
    for (int ee = 0; ee <= e; ++ee) {
      const int wend = (ee == e) ? warp : kSelWarps;
      for (int w = 0; w < wend; ++w) before += s.warp_cnt[ee][w];
    }
    before += __popc(ball[e] & ((1u << lane) - 1u));
    const bool keep = rank[e] < K;
    if (keep) {
      if (kept_b) kept_b[before] = i;
      if (prev_kept_b) prev_kept_b[before] = prev_b ? prev_b[i] : 1.0f;
    } else if (dropped_b) dropped_b[i - before] = i;
  }
}

__global__ void __launch_bounds__(kSelThreads)
select_topk_kernel(const float* __restrict__ score, int N, int K, int order,
                   int64_t* __restrict__ kept, int64_t* __restrict__ dropped) {
  __shared__ SelSmem s;
  const int b = blockIdx.x;
  for (int i = threadIdx.x; i < N; i += kSelThreads) s.key[i] = float_to_ordered(score[(size_t)b * N + i]);
  if (threadIdx.x < 4) s.key[N + threadIdx.x] = 0u;  // padding for the 4-wide rank loop
  __syncthreads();
  block_select_write(s, N, K, order, kept ? kept + (size_t)b * K : nullptr,
                     dropped ? dropped + (size_t)b * (N - K) : nullptr);
}

// ---- dynamic keep-ratio ("threshold") selection: the prefix-sum form of kernel (1) -------------------------------------------
// Reference: vit_models/dynamic_vit.py:880-890 (training) / :935-945 (inference): ascending sort of the keep probabilities,
// cumulative sum, keep the tokens whose cumulative mass exceeds the threshold, scatter the flags back to token order.
// One CTA per image: ascending stable rank by counting (same keys as the top-K select), the sorted values land in shared
// memory, ONE thread runs the prefix sum in index order with a double accumulator rounded to float per prefix -- exactly
// torch's CPU cumsum (acc_type<float> = double), the oracle's arithmetic -- and every token reads the prefix at its own rank.
// Outputs: mask (B,N) uint8 0/1 (a torch.bool tensor's storage), count (B) int32 = kept tokens per image, kept (B,N) int64 =
// the kept token indices in ascending order followed by -1 padding (the index list a varlen gather consumes); NULL to skip.
// kVar (d2s_threshold_select_varlen_f32): image b selects among its first nv[b] scores of the N-wide row (the rest is never read);
// mask / kept entries past nv[b] are 0 / -1.
template <bool kVar>
__global__ void __launch_bounds__(kSelThreads)
threshold_select_kernel(const float* __restrict__ score, int N, float threshold, uint8_t* __restrict__ mask,
                        int* __restrict__ count, int64_t* __restrict__ kept, const int* __restrict__ nv) {
  __shared__ SelSmem s;
  __shared__ float sorted_s[kSelMaxN];
  __shared__ int total_s;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int Nv = kVar ? min(max(nv[b], 0), N) : N;   // valid scores of this image; N is the row pitch
  if (kVar) {
    for (int i = Nv + tid; i < N; i += kSelThreads) {
      if (mask) mask[(size_t)b * N + i] = 0;
      if (kept) kept[(size_t)b * N + i] = -1;
    }
  }
  float myv[kSelEPT];
  uint32_t mykey[kSelEPT];
#pragma unroll
  for (int e = 0; e < kSelEPT; ++e) {
    const int i = e * kSelThreads + tid;
    myv[e] = (i < Nv) ? score[(size_t)b * N + i] : 0.f;
    mykey[e] = float_to_ordered(myv[e]);
    if (i < Nv) s.key[i] = mykey[e];
  }
  __syncthreads();
  int rank[kSelEPT];
#pragma unroll
  for (int e = 0; e < kSelEPT; ++e) rank[e] = 0;
  const int nchunks = (Nv + kSelThreads - 1) / kSelThreads;
  for (int j = 0; j < Nv; ++j) {
    const uint32_t kj = s.key[j];  // broadcast read
#pragma unroll
    for (int e = 0; e < kSelEPT; ++e)
      if (e < nchunks) rank[e] += (kj < mykey[e]) || (kj == mykey[e] && j < e * kSelThreads + tid);
  }
#pragma unroll
  for (int e = 0; e < kSelEPT; ++e)
    if (e * kSelThreads + tid < Nv) sorted_s[rank[e]] = myv[e];
  __syncthreads();
  if (tid == 0) {
    double acc = 0.0;
    for (int r = 0; r < Nv; ++r) {
      acc += (double)sorted_s[r];
      sorted_s[r] = (float)acc;
    }
  }
  __syncthreads();
  unsigned ball[kSelEPT];
#pragma unroll
  for (int e = 0; e < kSelEPT; ++e) {
    const int i = e * kSelThreads + tid;
    const bool keep = (i < Nv) && (sorted_s[rank[e]] > threshold);
    if (i < Nv && mask) mask[(size_t)b * N + i] = keep ? 1 : 0;
    ball[e] = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) s.warp_cnt[e][warp] = __popc(ball[e]);
  }
  __syncthreads();
  if (tid == 0) {
    int t = 0;
    for (int e = 0; e < nchunks; ++e)
      for (int w = 0; w < kSelWarps; ++w) t += s.warp_cnt[e][w];
    total_s = t;
    if (count) count[b] = t;
  }
  if (kept == nullptr) return;
  __syncthreads();
#pragma unroll
  for (int e = 0; e < kSelEPT; ++e) {
    const int i = e * kSelThreads + tid;
    if (i >= Nv) continue;
    int before = 0;
    for (int ee = 0; ee <= e; ++ee) {
      const int wend = (ee == e) ? warp : kSelWarps;
      for (int w = 0; w < wend; ++w) before += s.warp_cnt[ee][w];
    }
    before += __popc(ball[e] & ((1u << lane) - 1u));
    if ((ball[e] >> lane) & 1u) kept[(size_t)b * N + before] = i;
    else kept[(size_t)b * N + total_s + (i - before)] = -1;      // padding behind the kept list
  }
}

// ---- per-token dot products of the tails ---------------------------------------------------------
// One thread per token walks its C-element row with 16-byte loads (the row is contiguous; the warp's
// lines are all used and stay in L1 between consecutive loads).  Weights are broadcast from smem.
template <typename T_> struct Vec16;
template <> struct Vec16<float> {
  static constexpr int kElems = 4;
  __device__ static void load(const float* p, float (&v)[8]) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
};
template <> struct Vec16<__nv_bfloat16> {
  static constexpr int kElems = 8;
  __device__ static void load(const __nv_bfloat16* p, float (&v)[8]) {
    const uint4 t = *reinterpret_cast<const uint4*>(p);
    const uint32_t w[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
};

__device__ __forceinline__ float round_to(float f, const float*) { return f; }
__device__ __forceinline__ float round_to(float f, const __nv_bfloat16*) { return __bfloat162float(__float2bfloat16_rn(f)); }

__device__ __forceinline__ float block_reduce_max(float v, SelSmem& s) {
  v = warp_max(v);
  if ((threadIdx.x & 31) == 0) s.red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = s.red[0];
    for (int w = 1; w < kSelWarps; ++w) m = fmaxf(m, s.red[w]);
    s.bcast = m;
  }
  __syncthreads();
  const float r = s.bcast;
  __syncthreads();
  return r;
}
__device__ __forceinline__ float block_reduce_sum(float v, SelSmem& s) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) s.red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = 0.f;
    for (int w = 0; w < kSelWarps; ++w) m += s.red[w];
    s.bcast = m;
  }
  __syncthreads();
  const float r = s.bcast;
  __syncthreads();
  return r;
}

// Gumbel keep decision for one token.  Reference: torch F.gumbel_softmax(hard=True) over 2 classes,
// class 0 = keep: keep iff softmax(x)[0] >= softmax(x)[1] with x = logp + g, i.e. iff
// exp(x0 - max) >= exp(x1 - max).  For x0 < x1 that holds only when exp(x0 - x1) rounds to 1.0f.
__device__ __forceinline__ void gumbel_decide(float lp0, float lp1, float g0, float g1, float prev,
                                              float& decision, float& ysoft0) {
  const float x0 = __fadd_rn(lp0, g0), x1 = __fadd_rn(lp1, g1);
  const float m = fmaxf(x0, x1);
  const float e0 = expf(__fsub_rn(x0, m)), e1 = expf(__fsub_rn(x1, m));
  ysoft0 = e0 / (e0 + e1);
  decision = (e0 >= e1 ? 1.0f : 0.0f) * prev;
}

template <typename T_>
__global__ void __launch_bounds__(kSelThreads)
score_tail_a_kernel(const T_* __restrict__ hidden, int N, int C, const float* __restrict__ W,
                    const float* __restrict__ bias, int K, const float* __restrict__ gumbel,
                    const float* __restrict__ prev, float* __restrict__ logp, int64_t* __restrict__ kept,
                    float* __restrict__ decision, float* __restrict__ ysoft, int act_input, float* __restrict__ prev_kept) {
  __shared__ SelSmem s;
  extern __shared__ float w_s[];  // 2*C weights
  const int b = blockIdx.x;
  for (int i = threadIdx.x; i < 2 * C; i += kSelThreads) w_s[i] = W[i];
  __syncthreads();
  const float b0 = bias[0], b1 = bias[1];
  constexpr int VE = Vec16<T_>::kElems;
  // Four lanes per token row: lane q of a quad takes the 16-byte chunks q, q+4, q+8, ... of the row, so every load
  // instruction of the warp covers 8 rows x 64 contiguous bytes (all sectors fully used) instead of 32 rows x 16 bytes.
  const int quad = threadIdx.x >> 2, q4 = threadIdx.x & 3;
  const int nchunk = C / VE;
  for (int n0 = 0; n0 < N; n0 += kSelThreads / 4) {
    const int n = n0 + quad;
    float a0 = 0.f, a1 = 0.f;
    if (n < N) {
      const T_* row = hidden + ((size_t)b * N + n) * C;
      for (int ch = q4; ch < nchunk; ch += 4) {
        const int c = ch * VE;
        float v[8];
        Vec16<T_>::load(row + c, v);
        if (act_input) {  // the GELU in front of the last Linear (default_dynamic_vit.py:318), applied on load
#pragma unroll
          for (int q = 0; q < VE; q += 2) {
            if (sizeof(T_) == 2) {   // bf16 activations: the packed fp32x2 erfcx GELU of the GEMM epilogues (<= 0.07 bf16 ulp); erff made
              float g0, g1;          // this tail FP32-bound (19 M erff per launch at B = 1024)
              f2_unpack(gelu_erf_pair(f2_pack(v[q], v[q + 1])), g0, g1);
              v[q] = round_to(g0, row);
              v[q + 1] = round_to(g1, row);
            } else {
              v[q] = round_to(0.5f * v[q] * (1.0f + erff(v[q] * 0.70710678118654752440f)), row);
              v[q + 1] = round_to(0.5f * v[q + 1] * (1.0f + erff(v[q + 1] * 0.70710678118654752440f)), row);
            }
          }
        }
#pragma unroll
        for (int q = 0; q < VE; ++q) {
          a0 = fmaf(v[q], w_s[c + q], a0);
          a1 = fmaf(v[q], w_s[C + c + q], a1);
        }
      }
    }
    a0 += __shfl_xor_sync(0xffffffffu, a0, 1);
    a1 += __shfl_xor_sync(0xffffffffu, a1, 1);
    a0 += __shfl_xor_sync(0xffffffffu, a0, 2);
    a1 += __shfl_xor_sync(0xffffffffu, a1, 2);
    if (n < N && q4 == 0) {
      a0 += b0; a1 += b1;
      const float m = fmaxf(a0, a1);
      const float lse = m + logf(expf(a0 - m) + expf(a1 - m));
      const float lp0 = a0 - lse, lp1 = a1 - lse;
      const size_t t = (size_t)b * N + n;
      reinterpret_cast<float2*>(logp)[t] = make_float2(lp0, lp1);
      if (gumbel) {
        float d, y;
        const float2 g = reinterpret_cast<const float2*>(gumbel)[t];
        gumbel_decide(lp0, lp1, g.x, g.y, prev ? prev[t] : 1.0f, d, y);
        decision[t] = d;
        ysoft[t] = y;
      }
      s.key[n] = float_to_ordered(lp0);
    }
  }
  if (kept == nullptr) return;
  if (threadIdx.x < 4) s.key[N + threadIdx.x] = 0u;
  __syncthreads();
  block_select_write(s, N, K, D2S_ORDER_SCORE_DESC, kept + (size_t)b * K, nullptr, prev ? prev + (size_t)b * N : nullptr,
                     prev_kept ? prev_kept + (size_t)b * K : nullptr);
}

// kVar (d2s_score_tail_b_varlen): image b has nv[b] valid rows of its N (padded) rows; the softmax runs over those only, pad rows
// are never read, their scores are -inf and their probabilities 0 (no selection)
template <typename T_, bool kVar = false>
__global__ void __launch_bounds__(kSelThreads)
score_tail_b_kernel(const T_* __restrict__ hidden, int N, int C, const float* __restrict__ ln_w,
                    const float* __restrict__ ln_b, float ln_eps, const float* __restrict__ W,
                    const float* __restrict__ bias_p, int prob_mode, int K, float* __restrict__ scores, float* __restrict__ probs,
                    int64_t* __restrict__ kept, int64_t* __restrict__ dropped, const int* __restrict__ nv) {
  __shared__ SelSmem s;
  extern __shared__ float w_s[];  // gw[c] = ln_w[c]*W[c] (or W[c]),  then scalar sum(ln_b*W)
  const int b = blockIdx.x;
  const float bias = bias_p ? bias_p[0] : 0.f;
  float part = 0.f;
  for (int i = threadIdx.x; i < C; i += kSelThreads) {
    w_s[i] = ln_w ? ln_w[i] * W[i] : W[i];
    if (ln_w) part += ln_b[i] * W[i];
  }
  const float beta_dot = block_reduce_sum(part, s);  // also orders the w_s writes before use
  constexpr int VE = Vec16<T_>::kElems;
  constexpr int kMaxPerThread = kSelEPT;
  // Phase 1 (four lanes per token row, see score_tail_a_kernel): raw scores into shared memory.
  const int quad = threadIdx.x >> 2, q4 = threadIdx.x & 3;
  const int nchunk = C / VE;
  const int Nv = kVar ? min(max(nv[b], 0), N) : N;   // valid rows of this image; N is the row pitch
  float* sc_s = reinterpret_cast<float*>(s.key);   // scores live in the key array until they are turned into keys
  for (int n0 = 0; n0 < Nv; n0 += kSelThreads / 4) {
    const int n = n0 + quad;
    const T_* row = hidden + ((size_t)b * N + min(n, Nv - 1)) * C;
    float mean = 0.f, rstd = 1.f;
    if (ln_w) {
      float sum = 0.f;
      for (int ch = q4; ch < nchunk; ch += 4) {
        float v[8];
        Vec16<T_>::load(row + ch * VE, v);
#pragma unroll
        for (int q = 0; q < VE; ++q) sum += v[q];
      }
      sum += __shfl_xor_sync(0xffffffffu, sum, 1);
      sum += __shfl_xor_sync(0xffffffffu, sum, 2);
      mean = sum / (float)C;
    }
    float var = 0.f, dot = 0.f;
    for (int ch = q4; ch < nchunk; ch += 4) {   // second touch of the row hits L1 (8 rows x 192 B per warp pass)
      const int c = ch * VE;
      float v[8];
      Vec16<T_>::load(row + c, v);
#pragma unroll
      for (int q = 0; q < VE; ++q) {
        const float d = v[q] - mean;
        var = fmaf(d, d, var);
        dot = fmaf(d, w_s[c + q], dot);
      }
    }
    var += __shfl_xor_sync(0xffffffffu, var, 1);
    dot += __shfl_xor_sync(0xffffffffu, dot, 1);
    var += __shfl_xor_sync(0xffffffffu, var, 2);
    dot += __shfl_xor_sync(0xffffffffu, dot, 2);
    if (ln_w) rstd = rsqrtf(var / (float)C + ln_eps);
    if (n < Nv && q4 == 0) {
      const float val = dot * rstd + beta_dot + bias;
      sc_s[n] = val;
      scores[(size_t)b * N + n] = val;
    }
  }
  __syncthreads();
  float sc[kMaxPerThread];
  float lmax = -INFINITY;
#pragma unroll
  for (int e = 0; e < kMaxPerThread; ++e) {
    const int n = e * kSelThreads + threadIdx.x;
    sc[e] = (n < Nv) ? sc_s[n] : -INFINITY;
    lmax = fmaxf(lmax, sc[e]);
  }
  __syncthreads();   // every score has been read before the key array is overwritten below
  float pr[kMaxPerThread];
  if (prob_mode == D2S_PROB_SOFTMAX) {
    const float gmax = block_reduce_max(lmax, s);
    float lsum = 0.f;
#pragma unroll
    for (int e = 0; e < kMaxPerThread; ++e) {
      const int n = e * kSelThreads + threadIdx.x;
      pr[e] = (n < Nv) ? expf(sc[e] - gmax) : 0.f;
      lsum += pr[e];
    }
    const float gsum = block_reduce_sum(lsum, s);
#pragma unroll
    for (int e = 0; e < kMaxPerThread; ++e) pr[e] = pr[e] / gsum;
  } else {
#pragma unroll
    for (int e = 0; e < kMaxPerThread; ++e) pr[e] = 1.0f / (1.0f + expf(-sc[e]));
  }
#pragma unroll
  for (int e = 0; e < kMaxPerThread; ++e) {
    const int n = e * kSelThreads + threadIdx.x;
    if (n < Nv) {
      probs[(size_t)b * N + n] = pr[e];
      s.key[n] = float_to_ordered(pr[e]);
    } else if (kVar && n < N) {
      probs[(size_t)b * N + n] = 0.f;
      scores[(size_t)b * N + n] = -INFINITY;
    }
  }
  if (kept == nullptr) return;
  if (threadIdx.x < 4) s.key[N + threadIdx.x] = 0u;
  __syncthreads();
  block_select_write(s, N, K, D2S_ORDER_INDEX_ASC, kept + (size_t)b * K,
                     dropped ? dropped + (size_t)b * (N - K) : nullptr);
}

__global__ void gumbel_decision_kernel(const float* __restrict__ logp, const float* __restrict__ gumbel,
                                       const float* __restrict__ prev, int64_t n, float* __restrict__ decision,
                                       float* __restrict__ ysoft) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
    const float2 lp = reinterpret_cast<const float2*>(logp)[t];
    const float2 g = reinterpret_cast<const float2*>(gumbel)[t];
    float d, y;
    gumbel_decide(lp.x, lp.y, g.x, g.y, prev ? prev[t] : 1.0f, d, y);
    decision[t] = d;
    if (ysoft) ysoft[t] = y;
  }
}

// Straight-through backward: value = (hard - y.detach() + y)[0] * prev, so
//   d/dlogp = (+g, -g) with g = gout * prev * y0 * (1 - y0)      (only y_soft carries gradient)
//   d/dprev = gout * hard0                                        (prev is the previous stage's decision, :459)
// hard0 and y0 are recomputed from (logp, gumbel) with the forward's own routine: bit-identical, nothing saved.
__global__ void gumbel_decision_bwd_kernel(const float* __restrict__ gout, const float* __restrict__ logp,
                                           const float* __restrict__ gumbel, const float* __restrict__ prev, int64_t n,
                                           float* __restrict__ glogp, float* __restrict__ gprev) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
    const float2 lp = reinterpret_cast<const float2*>(logp)[t];
    const float2 gm = reinterpret_cast<const float2*>(gumbel)[t];
    float hard0, y;
    gumbel_decide(lp.x, lp.y, gm.x, gm.y, 1.0f, hard0, y);
    const float go = gout[t];
    const float g = go * (prev ? prev[t] : 1.0f) * y * (1.0f - y);
    reinterpret_cast<float2*>(glogp)[t] = make_float2(g, -g);
    if (gprev) gprev[t] = go * hard0;
  }
}

static int grid_1d(int64_t n, int threads) {
  int64_t blocks = (n + threads - 1) / threads;
  const int64_t cap = 8LL * kNumSMs;
  return (int)(blocks < cap ? (blocks < 1 ? 1 : blocks) : cap);
}

}  // namespace d2s

using namespace d2s;

extern "C" int d2s_select_topk_f32(const float* score, int B, int N, int K, int order, int64_t* kept,
                                   int64_t* dropped, d2s_stream_t stream) {
  D2S_REQUIRE(score && (kept || dropped), D2S_ERR_ARG, "select: null pointer");
  D2S_REQUIRE(B >= 0 && N >= 1 && N <= kSelMaxN, D2S_ERR_ARG, "select: N=%d outside [1,%d]", N, kSelMaxN);
  D2S_REQUIRE(K >= 0 && K <= N, D2S_ERR_ARG, "select: K=%d outside [0,N=%d]", K, N);
  D2S_REQUIRE(order == D2S_ORDER_INDEX_ASC || order == D2S_ORDER_SCORE_DESC, D2S_ERR_ARG, "select: bad order %d", order);
  if (B == 0) return D2S_OK;
  select_topk_kernel<<<B, kSelThreads, 0, (cudaStream_t)stream>>>(score, N, K, order, kept, dropped);
  count_launch();
  return check_launch("d2s_select_topk_f32");
}

extern "C" int d2s_threshold_select_f32(const float* score, int B, int N, float threshold, uint8_t* mask, int* count,
                                       int64_t* kept, d2s_stream_t stream) {
  D2S_REQUIRE(score && (mask || kept || count), D2S_ERR_ARG, "threshold_select: null pointer");
  D2S_REQUIRE(B >= 0 && N >= 1 && N <= kSelMaxN, D2S_ERR_ARG, "threshold_select: N=%d outside [1,%d]", N, kSelMaxN);
  if (B == 0) return D2S_OK;
  threshold_select_kernel<false><<<B, kSelThreads, 0, (cudaStream_t)stream>>>(score, N, threshold, mask, count, kept, nullptr);
  count_launch();
  return check_launch("d2s_threshold_select_f32");
}

extern "C" int d2s_threshold_select_varlen_f32(const float* score, const int* n, int B, int Nmax, float threshold, uint8_t* mask,
                                              int* count, int64_t* kept, d2s_stream_t stream) {
  D2S_REQUIRE(score && n && (mask || kept || count), D2S_ERR_ARG, "threshold_select_varlen: null pointer");
  D2S_REQUIRE(B >= 0 && Nmax >= 1 && Nmax <= kSelMaxN, D2S_ERR_ARG, "threshold_select_varlen: Nmax=%d outside [1,%d]", Nmax, kSelMaxN);
  if (B == 0) return D2S_OK;
  threshold_select_kernel<true><<<B, kSelThreads, 0, (cudaStream_t)stream>>>(score, Nmax, threshold, mask, count, kept, n);
  count_launch();
  return check_launch("d2s_threshold_select_varlen_f32");
}

static int check_tail(const void* hidden, int dtype, int B, int N, int C, int K) {
  D2S_REQUIRE(hidden, D2S_ERR_ARG, "score_tail: null hidden");
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "score_tail: dtype %d unsupported", dtype);
  D2S_REQUIRE(B >= 0 && N >= 1 && N <= kSelMaxN, D2S_ERR_ARG, "score_tail: N=%d outside [1,%d]", N, kSelMaxN);
  D2S_REQUIRE(C >= 8 && C <= 1024 && C % 8 == 0, D2S_ERR_ARG, "score_tail: C=%d must be a multiple of 8 in [8,1024]", C);
  D2S_REQUIRE(K >= 0 && K <= N, D2S_ERR_ARG, "score_tail: K=%d outside [0,N=%d]", K, N);
  D2S_REQUIRE(aligned16(hidden), D2S_ERR_ALIGN, "score_tail: hidden must be 16-byte aligned");
  return D2S_OK;
}

extern "C" int d2s_score_tail_a(const void* hidden, int dtype, int B, int N, int C, const float* W,
                                const float* bias, int K, const float* gumbel, const float* prev, float* logp,
                                int64_t* kept, float* decision, float* ysoft, int act_input, float* prev_kept,
                                d2s_stream_t stream) {
  int rc = check_tail(hidden, dtype, B, N, C, K);
  if (rc) return rc;
  D2S_REQUIRE(W && bias && logp, D2S_ERR_ARG, "score_tail_a: null W/bias/logp");
  D2S_REQUIRE(!gumbel || (decision && ysoft), D2S_ERR_ARG, "score_tail_a: gumbel given without decision/ysoft outputs");
  D2S_REQUIRE(!prev_kept || kept, D2S_ERR_ARG, "score_tail_a: prev_kept needs kept");
  D2S_REQUIRE(act_input == D2S_ACT_NONE || act_input == D2S_ACT_GELU, D2S_ERR_ARG, "score_tail_a: bad act_input %d", act_input);
  if (B == 0) return D2S_OK;
  const size_t smem = 2 * (size_t)C * sizeof(float);
  if (dtype == D2S_F32)
    score_tail_a_kernel<float><<<B, kSelThreads, smem, (cudaStream_t)stream>>>(
        (const float*)hidden, N, C, W, bias, K, gumbel, prev, logp, kept, decision, ysoft, act_input, prev_kept);
  else
    score_tail_a_kernel<__nv_bfloat16><<<B, kSelThreads, smem, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)hidden, N, C, W, bias, K, gumbel, prev, logp, kept, decision, ysoft, act_input, prev_kept);
  count_launch();
  return check_launch("d2s_score_tail_a");
}

extern "C" int d2s_score_tail_b(const void* hidden, int dtype, int B, int N, int C, const float* ln_w,
                                const float* ln_b, float ln_eps, const float* W, const float* bias, int prob_mode, int K,
                                float* scores, float* probs, int64_t* kept, int64_t* dropped, d2s_stream_t stream) {
  int rc = check_tail(hidden, dtype, B, N, C, K);
  if (rc) return rc;
  D2S_REQUIRE(W && scores && probs, D2S_ERR_ARG, "score_tail_b: null W/scores/probs");
  D2S_REQUIRE((ln_w == nullptr) == (ln_b == nullptr), D2S_ERR_ARG, "score_tail_b: ln_w and ln_b must both be set or both NULL");
  D2S_REQUIRE(prob_mode == D2S_PROB_SOFTMAX || prob_mode == D2S_PROB_SIGMOID, D2S_ERR_ARG, "score_tail_b: bad prob_mode");
  D2S_REQUIRE(kept || !dropped, D2S_ERR_ARG, "score_tail_b: dropped without kept");
  if (B == 0) return D2S_OK;
  const size_t smem = (size_t)C * sizeof(float);
  if (dtype == D2S_F32)
    score_tail_b_kernel<float><<<B, kSelThreads, smem, (cudaStream_t)stream>>>(
        (const float*)hidden, N, C, ln_w, ln_b, ln_eps, W, bias, prob_mode, K, scores, probs, kept, dropped, nullptr);
  else
    score_tail_b_kernel<__nv_bfloat16><<<B, kSelThreads, smem, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)hidden, N, C, ln_w, ln_b, ln_eps, W, bias, prob_mode, K, scores, probs, kept, dropped, nullptr);
  count_launch();
  return check_launch("d2s_score_tail_b");
}

extern "C" int d2s_score_tail_b_varlen(const void* hidden, const int* n, int dtype, int B, int Nmax, int C, const float* ln_w,
                                       const float* ln_b, float ln_eps, const float* W, const float* bias, int prob_mode, float* scores,
                                       float* probs, d2s_stream_t stream) {
  D2S_REQUIRE(n, D2S_ERR_ARG, "score_tail_b_varlen: null n");
  int rc = check_tail(hidden, dtype, B, Nmax, C, 0);
  if (rc) return rc;
  D2S_REQUIRE(W && scores && probs, D2S_ERR_ARG, "score_tail_b_varlen: null W/scores/probs");
  D2S_REQUIRE((ln_w == nullptr) == (ln_b == nullptr), D2S_ERR_ARG, "score_tail_b_varlen: ln_w and ln_b must both be set or both NULL");
  D2S_REQUIRE(prob_mode == D2S_PROB_SOFTMAX || prob_mode == D2S_PROB_SIGMOID, D2S_ERR_ARG, "score_tail_b_varlen: bad prob_mode");
  if (B == 0) return D2S_OK;
  const size_t smem = (size_t)C * sizeof(float);
  if (dtype == D2S_F32)
    score_tail_b_kernel<float, true><<<B, kSelThreads, smem, (cudaStream_t)stream>>>(
        (const float*)hidden, Nmax, C, ln_w, ln_b, ln_eps, W, bias, prob_mode, 0, scores, probs, nullptr, nullptr, n);
  else
    score_tail_b_kernel<__nv_bfloat16, true><<<B, kSelThreads, smem, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)hidden, Nmax, C, ln_w, ln_b, ln_eps, W, bias, prob_mode, 0, scores, probs, nullptr, nullptr, n);
  count_launch();
  return check_launch("d2s_score_tail_b_varlen");
}

extern "C" int d2s_gumbel_decision_f32(const float* logp, const float* gumbel, const float* prev, int64_t n,
                                       float* decision, float* ysoft, d2s_stream_t stream) {
  D2S_REQUIRE(logp && gumbel && decision, D2S_ERR_ARG, "gumbel_decision: null pointer");
  D2S_REQUIRE(n >= 0, D2S_ERR_ARG, "gumbel_decision: n < 0");
  if (n == 0) return D2S_OK;
  gumbel_decision_kernel<<<grid_1d(n, 256), 256, 0, (cudaStream_t)stream>>>(logp, gumbel, prev, n, decision, ysoft);
  count_launch();
  return check_launch("d2s_gumbel_decision_f32");
}

extern "C" int d2s_gumbel_decision_bwd_f32(const float* gout, const float* logp, const float* gumbel, const float* prev,
                                           int64_t n, float* glogp, float* gprev, d2s_stream_t stream) {
  D2S_REQUIRE(gout && logp && gumbel && glogp, D2S_ERR_ARG, "gumbel_decision_bwd: null pointer");
  D2S_REQUIRE(n >= 0, D2S_ERR_ARG, "gumbel_decision_bwd: n < 0");
  if (n == 0) return D2S_OK;
  gumbel_decision_bwd_kernel<<<grid_1d(n, 256), 256, 0, (cudaStream_t)stream>>>(gout, logp, gumbel, prev, n, glogp, gprev);
  count_launch();
  return check_launch("d2s_gumbel_decision_bwd_f32");
}
