// Predictor body helpers (inference path of PredictorLG.forward, vit_models/default_dynamic_vit.py:324-330 and
// dynamic_vit.py:538-546): the reference runs GELU, a policy multiply, two reductions, a division, an expand and a
// concat as separate passes over the (B,N,C) activations.  Here:
//
//   pool_act_kernel : one pass over z = in_conv's Linear output.  local = act(z[:, :, :C/2]) is written densely as the
//                     A operand of the next Linear; pooled[b] = sum_n act(z[b,n,C/2:]) * policy[b,n] / sum_n policy[b,n]
//                     (policy NULL => plain mean, dynamic_vit.py:542) never leaves the chip as a (B,N,C/2) tensor.
//   bias_act_kernel : u = act(u + bias[b]) in place with a PER-IMAGE bias row.  With the next Linear split as
//                     W = [W_local | W_global], Linear(cat(local, pooled)) = local @ W_local^T + (pooled @ W_global^T + b),
//                     so the concat (default_dynamic_vit.py:329) is never materialised.
//
// Both are HBM-bound: pool_act reads e*N*C and writes e*N*C/2 per image, bias_act reads and writes e*N*C' once.
#include "d2s_tc.cuh"

namespace d2s {

template <typename T_> struct PVec;
template <> struct PVec<__nv_bfloat16> {
  static constexpr int kElems = 8;
  __device__ static void unpack(const int4& r, float (&v)[8]) {
    const uint32_t w[4] = {(uint32_t)r.x, (uint32_t)r.y, (uint32_t)r.z, (uint32_t)r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  __device__ static int4 pack(const float (&v)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<const uint32_t*>(&t);
    }
    return make_int4((int)w[0], (int)w[1], (int)w[2], (int)w[3]);
  }
  __device__ static float round(float f) { return __bfloat162float(__float2bfloat16_rn(f)); }
};
template <> struct PVec<float> {
  static constexpr int kElems = 4;
  __device__ static void unpack(const int4& r, float (&v)[8]) {
    v[0] = __int_as_float(r.x); v[1] = __int_as_float(r.y); v[2] = __int_as_float(r.z); v[3] = __int_as_float(r.w);
  }
  __device__ static int4 pack(const float (&v)[8]) {
    return make_int4(__float_as_int(v[0]), __float_as_int(v[1]), __float_as_int(v[2]), __float_as_int(v[3]));
  }
  __device__ static float round(float f) { return f; }
};

// erf for activations that are stored as bf16: Abramowitz-Stegun 7.1.26 (|error| <= 1.5e-7 with exact exp) evaluated with
// MUFU rcp/ex2 -- absolute error ~5e-7, three orders of magnitude below half a bf16 ulp of the GELU it feeds, at
// roughly a third of erff()'s instruction count (exact-erf GELU is COMPUTE-bound on B200: ~30 FP32 instructions per
// element against 4 bytes of traffic).  fp32 tensors keep erff().
// Returns 1 + erf(x).  For x < 0 this is erfc(|x|) = p*e directly (no cancellation in the GELU's negative tail).
__device__ __forceinline__ float one_plus_erf_fast(float x) {
  const float ax = fabsf(x);
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, ax, 1.0f)));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  p *= t;
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * ax * ax));
  const float pe = p * e;
  return x < 0.f ? pe : 2.0f - pe;
}
template <bool kFast>
__device__ __forceinline__ float act_apply(float x, int act) {
  if (act == D2S_ACT_GELU) {   // nn.GELU() (erf form)
    const float z = x * 0.70710678118654752440f;
    return 0.5f * x * (kFast ? one_plus_erf_fast(z) : 1.0f + erff(z));
  }
  if (act == D2S_ACT_RELU) return fmaxf(x, 0.0f);
  return x;
}
template <typename T_> struct ActFast { static constexpr bool value = false; };
template <> struct ActFast<__nv_bfloat16> { static constexpr bool value = true; };

constexpr int kPoolThreads = 256;

// grid = B; thread = (16-byte vector column v, token group g); groups stride the tokens
template <typename T_>
__global__ void __launch_bounds__(kPoolThreads)
pool_act_kernel(const T_* __restrict__ z, const float* __restrict__ policy, int N, int C, int act,
                T_* __restrict__ local, T_* __restrict__ pooled, long long zbs) {
  constexpr int VE = PVec<T_>::kElems;
  extern __shared__ float red[];  // groups x (C/2) partial sums, then groups partial policy sums
  const int b = blockIdx.x;
  const int nvec = C / VE, half_vec = nvec / 2, half = C / 2;
  // local == NULL: only the pooled global half is wanted (z is already activated and its local half is consumed in place
  // by the next kernel): the threads cover the upper half of the row only, twice as many token groups
  const bool only_pool = local == nullptr;
  const int tv = only_pool ? half_vec : nvec;          // 16-byte vectors per token row handled here
  const int groups = kPoolThreads / tv;                // host guarantees nvec <= kPoolThreads
  const int v = (only_pool ? half_vec : 0) + threadIdx.x % tv, g = threadIdx.x / tv;
  float acc[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) acc[q] = 0.f;
  float psum = 0.f;
  if (g < groups) {
    // bf16 GELU here goes through the packed fp32x2 erfcx polynomial of the GEMM epilogues (d2s_tc.cuh gelu_erf_pair, <= 0.07
    // bf16 ulp, one MUFU and ~10 issue slots per element): with the rcp-based erf this kernel was bound by the FP32 pipe.
    auto token = [&](int n, const int4& raw) {
      const size_t row = (size_t)b * N + n;
      float x[8];
      PVec<T_>::unpack(raw, x);
      if (ActFast<T_>::value && act == D2S_ACT_GELU) {
#pragma unroll
        for (int q = 0; q < VE; q += 2) f2_unpack(gelu_erf_pair(f2_pack(x[q], x[q + 1])), x[q], x[q + 1]);
      } else {
#pragma unroll
        for (int q = 0; q < VE; ++q) x[q] = act_apply<false>(x[q], act);
      }
#pragma unroll
      for (int q = 0; q < VE; ++q) x[q] = PVec<T_>::round(x[q]);
      if (v < half_vec) {
        *reinterpret_cast<int4*>(local + row * half + (size_t)v * VE) = PVec<T_>::pack(x);
      } else {
        const float p = policy ? policy[row] : 1.0f;
#pragma unroll
        for (int q = 0; q < VE; ++q) acc[q] = fmaf(x[q], p, acc[q]);
        if (v == half_vec) psum += p;
      }
    };
    const T_* zb = z + (size_t)b * zbs + (size_t)v * VE;          // zbs: elements between images (N * C when dense)
    int n = g;
    for (; n + 3 * groups < N; n += 4 * groups) {      // four token rows in flight per thread
      const int4 r0 = ld_stream16(zb + (size_t)n * C);
      const int4 r1 = ld_stream16(zb + (size_t)(n + groups) * C);
      const int4 r2 = ld_stream16(zb + (size_t)(n + 2 * groups) * C);
      const int4 r3 = ld_stream16(zb + (size_t)(n + 3 * groups) * C);
      token(n, r0); token(n + groups, r1); token(n + 2 * groups, r2); token(n + 3 * groups, r3);
    }
    for (; n < N; n += groups) token(n, ld_stream16(zb + (size_t)n * C));
  }
  float* pol_red = red + (size_t)groups * half;
  if (g < groups && v >= half_vec) {
#pragma unroll
    for (int q = 0; q < VE; ++q) red[(size_t)g * half + (size_t)(v - half_vec) * VE + q] = acc[q];
    if (v == half_vec) pol_red[g] = psum;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < half; c += kPoolThreads) {
    float s = 0.f, ps = 0.f;
    for (int gg = 0; gg < groups; ++gg) { s += red[(size_t)gg * half + c]; ps += pol_red[gg]; }
    st_from_float(pooled, (size_t)b * half + c, s / ps);
  }
}

// In-place form for Variant B (dynamic_vit.py:538-545): z (B,N,C) already activated; the upper half of every token
// row is REPLACED by the image's mean over tokens of that upper half, i.e. z becomes cat(local, global.expand) without
// a second tensor.  grid = B; phase 1 reduces, phase 2 broadcasts.
// kVar (d2s_pool_concat_varlen_inplace): image b has Nv = nv[b] valid rows of its N (padded) rows; the mean runs over those and
// is written into those; pad rows are neither read nor written.
template <typename T_, bool kVar = false>
__global__ void __launch_bounds__(kPoolThreads)
pool_concat_inplace_kernel(T_* __restrict__ z, int N, int C, const int* __restrict__ nv) {
  constexpr int VE = PVec<T_>::kElems;
  extern __shared__ float red[];  // groups x (C/2), then the pooled row at red[0 .. C/2)
  const int b = blockIdx.x;
  const int Nv = kVar ? min(max(nv[b], 0), N) : N;
  const int hvec = C / VE / 2, half = C / 2;
  const int groups = kPoolThreads / hvec;   // host guarantees hvec <= kPoolThreads
  const int v = threadIdx.x % hvec, g = threadIdx.x / hvec;
  float acc[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) acc[q] = 0.f;
  if (g < groups) {
    for (int n = g; n < Nv; n += groups) {
      float x[8];
      PVec<T_>::unpack(*reinterpret_cast<const int4*>(z + ((size_t)b * N + n) * C + half + (size_t)v * VE), x);
#pragma unroll
      for (int q = 0; q < VE; ++q) acc[q] += x[q];
    }
#pragma unroll
    for (int q = 0; q < VE; ++q) red[(size_t)g * half + (size_t)v * VE + q] = acc[q];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < half; c += kPoolThreads) {
    float s = 0.f;
    for (int gg = 0; gg < groups; ++gg) s += red[(size_t)gg * half + c];
    red[(size_t)groups * half + c] = PVec<T_>::round(s / (float)Nv);  // torch.mean rounds to the tensor dtype
  }
  __syncthreads();
  if (g < groups) {
    float m[8];
#pragma unroll
    for (int q = 0; q < VE; ++q) m[q] = red[(size_t)groups * half + (size_t)v * VE + q];
    const int4 packed = PVec<T_>::pack(m);
    for (int n = g; n < Nv; n += groups)
      *reinterpret_cast<int4*>(z + ((size_t)b * N + n) * C + half + (size_t)v * VE) = packed;
  }
}

// u (rows, C) += bias (per image: bias[(row / N) * C + c]; N == 0 => one shared row; NULL => none), then act, in place.
// One CTA per block of kBiasRows rows, its 16-byte vectors dealt flat to the threads (every lane busy whatever C is), two
// vectors in flight per thread; the one 64-bit division (first image of the block) is done once per CTA.
constexpr int kBiasRows = 64;
template <typename T_>
__global__ void __launch_bounds__(256)
bias_act_kernel(T_* __restrict__ u, const T_* __restrict__ bias, long long rows, int N, int C, int act) {
  constexpr int VE = PVec<T_>::kElems;
  const int nvec = C / VE;
  const long long row0 = (long long)blockIdx.x * kBiasRows;
  const int nrows = (int)min((long long)kBiasRows, rows - row0);
  const int items = nrows * nvec;
  const long long img0 = N > 0 ? row0 / N : 0;
  const int rem0 = N > 0 ? (int)(row0 - img0 * N) : 0;
  T_* base = u + row0 * C;
  auto bias_of = [&](int i, float (&bv)[8]) {
    const int r = i / nvec, v = i - r * nvec;
    const long long img = N > 0 ? img0 + (rem0 + r) / N : 0;
    PVec<T_>::unpack(*reinterpret_cast<const int4*>(bias + img * C + (size_t)v * VE), bv);
  };
  auto finish = [&](int i, const int4& raw) {
    float x[8];
    PVec<T_>::unpack(raw, x);
    if (bias) {
      float bv[8];
      bias_of(i, bv);
#pragma unroll
      for (int q = 0; q < VE; ++q) x[q] = PVec<T_>::round(x[q] + bv[q]);
    }
    if (ActFast<T_>::value && act == D2S_ACT_GELU) {   // packed fp32x2 erfcx polynomial (d2s_tc.cuh), as in pool_act and the GEMM epilogues
#pragma unroll
      for (int q = 0; q < VE; q += 2) f2_unpack(gelu_erf_pair(f2_pack(x[q], x[q + 1])), x[q], x[q + 1]);
    } else {
#pragma unroll
      for (int q = 0; q < VE; ++q) x[q] = act_apply<false>(x[q], act);
    }
    reinterpret_cast<int4*>(base)[i] = PVec<T_>::pack(x);
  };
  int i = threadIdx.x;
  for (; i + 256 < items; i += 512) {
    const int4 r0 = reinterpret_cast<const int4*>(base)[i];
    const int4 r1 = reinterpret_cast<const int4*>(base)[i + 256];
    finish(i, r0);
    finish(i + 256, r1);
  }
  if (i < items) finish(i, reinterpret_cast<const int4*>(base)[i]);
}

// flat variant for bias == NULL: the tensor is one long vector array
template <typename T_>
__global__ void __launch_bounds__(256)
act_flat_kernel(T_* __restrict__ u, long long nvec_total, int act) {
  constexpr int VE = PVec<T_>::kElems;
  int4* p = reinterpret_cast<int4*>(u);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nvec_total; i += 2 * stride) {
    const bool two = i + stride < nvec_total;
    float x[8], y[8];
    const int4 a = p[i];
    int4 b = make_int4(0, 0, 0, 0);
    if (two) b = p[i + stride];
    PVec<T_>::unpack(a, x);
    PVec<T_>::unpack(b, y);
#pragma unroll
    for (int q = 0; q < VE; ++q) { x[q] = act_apply<ActFast<T_>::value>(x[q], act); y[q] = act_apply<ActFast<T_>::value>(y[q], act); }
    p[i] = PVec<T_>::pack(x);
    if (two) p[i + stride] = PVec<T_>::pack(y);
  }
}


// ---- training form of the predictors' local / global split (PredictorLG.forward, default_dynamic_vit.py:326-329 with the keep
// policy, dynamic_vit.py:541-545 with a plain mean) as one kernel each way instead of slice, multiply, sum, divide, expand, cat
// and their six autograd nodes:
//     out[b, n, :half] = h[b, n, :half]            pooled[b, c] = sum_n w[b, n] h[b, n, half + c] / sum_n w[b, n]
//     out[b, n, half + c] = pooled[b, c]           (w = policy, or 1 when policy is NULL)
// backward, with G[b, c] = sum_n dout[b, n, half + c] and S = sum_n w[b, n]:
//     dh[b, n, :half] = dout[b, n, :half]          dh[b, n, half + c] = w[b, n] G[b, c] / S
//     dpolicy[b, n] = sum_c (h[b, n, half + c] - pooled[b, c]) G[b, c] / S
// One CTA per image; a warp owns a row at a time (lane l: 16-byte vectors l, l + 32, .. of the half row), so the per-row dot
// product of the backward is a warp reduction.  Sums in fp32, one rounding at the end.
constexpr int kPtWarps = 8;
constexpr int kPtMaxK = 3;          // half-row vectors per lane: C/2 <= 3 * 32 * (8 | 4) elements

template <typename T_>
__global__ void __launch_bounds__(kPtWarps * 32)
pool_concat_fwd_kernel(const T_* __restrict__ h, const float* __restrict__ policy, int N, int C, T_* __restrict__ out,
                       float* __restrict__ pooled, float* __restrict__ wsum) {
  constexpr int VE = PVec<T_>::kElems;
  extern __shared__ float pt_red[];          // kPtWarps x half partial sums, then the pooled row in slot 0
  __shared__ float ws_red[kPtWarps];
  const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int half = C / 2, hvec = half / VE;
  const T_* hb = h + (size_t)b * N * C;
  T_* ob = out + (size_t)b * N * C;
  float acc[kPtMaxK][8];
#pragma unroll
  for (int k = 0; k < kPtMaxK; ++k)
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[k][q] = 0.f;
  float ws = 0.f;
  for (int n = warp; n < N; n += kPtWarps) {
    const float w = policy ? policy[(size_t)b * N + n] : 1.f;
    ws += w;
#pragma unroll
    for (int k = 0; k < kPtMaxK; ++k) {
      const int v = lane + 32 * k;
      if (v < hvec) {
        const int4 loc = *reinterpret_cast<const int4*>(hb + (size_t)n * C + (size_t)v * VE);
        const int4 glo = *reinterpret_cast<const int4*>(hb + (size_t)n * C + half + (size_t)v * VE);
        *reinterpret_cast<int4*>(ob + (size_t)n * C + (size_t)v * VE) = loc;
        float x[8];
        PVec<T_>::unpack(glo, x);
#pragma unroll
        for (int q = 0; q < VE; ++q) acc[k][q] = fmaf(w, x[q], acc[k][q]);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < kPtMaxK; ++k) {
    const int v = lane + 32 * k;
    if (v < hvec) {
#pragma unroll
      for (int q = 0; q < VE; ++q) pt_red[(size_t)warp * half + (size_t)v * VE + q] = acc[k][q];
    }
  }
  if (lane == 0) ws_red[warp] = ws;          // every lane of a warp holds the same row-weight sum
  __syncthreads();
  float S = 0.f;
#pragma unroll
  for (int w = 0; w < kPtWarps; ++w) S += ws_red[w];
  __syncthreads();
  for (int c = threadIdx.x; c < half; c += kPtWarps * 32) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kPtWarps; ++w) t += pt_red[(size_t)w * half + c];
    t /= S;
    pooled[(size_t)b * half + c] = t;
    pt_red[(size_t)kPtWarps * half + c] = t;
  }
  if (threadIdx.x == 0) wsum[b] = S;
  __syncthreads();
  int4 packed[kPtMaxK];
#pragma unroll
  for (int k = 0; k < kPtMaxK; ++k) {
    const int v = lane + 32 * k;
    if (v < hvec) {
      float m[8];
#pragma unroll
      for (int q = 0; q < VE; ++q) m[q] = pt_red[(size_t)kPtWarps * half + (size_t)v * VE + q];
      packed[k] = PVec<T_>::pack(m);
    }
  }
  for (int n = warp; n < N; n += kPtWarps)
#pragma unroll
    for (int k = 0; k < kPtMaxK; ++k) {
      const int v = lane + 32 * k;
      if (v < hvec) *reinterpret_cast<int4*>(ob + (size_t)n * C + half + (size_t)v * VE) = packed[k];
    }
}

template <typename T_>
__global__ void __launch_bounds__(kPtWarps * 32)
pool_concat_bwd_kernel(const T_* __restrict__ dout, const T_* __restrict__ h, const float* __restrict__ policy,
                       const float* __restrict__ pooled, const float* __restrict__ wsum, int N, int C, T_* __restrict__ dh,
                       float* __restrict__ dpolicy) {
  constexpr int VE = PVec<T_>::kElems;
  extern __shared__ float pt_red[];          // kPtWarps x half partial sums, then G / S in slot kPtWarps
  const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int half = C / 2, hvec = half / VE;
  const T_* gb = dout + (size_t)b * N * C;
  const T_* hb = h + (size_t)b * N * C;
  T_* db = dh + (size_t)b * N * C;
  float acc[kPtMaxK][8];
#pragma unroll
  for (int k = 0; k < kPtMaxK; ++k)
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[k][q] = 0.f;
  for (int n = warp; n < N; n += kPtWarps) {
#pragma unroll
    for (int k = 0; k < kPtMaxK; ++k) {
      const int v = lane + 32 * k;
      if (v < hvec) {
        const int4 loc = *reinterpret_cast<const int4*>(gb + (size_t)n * C + (size_t)v * VE);
        const int4 glo = *reinterpret_cast<const int4*>(gb + (size_t)n * C + half + (size_t)v * VE);
        *reinterpret_cast<int4*>(db + (size_t)n * C + (size_t)v * VE) = loc;
        float x[8];
        PVec<T_>::unpack(glo, x);
#pragma unroll
        for (int q = 0; q < VE; ++q) acc[k][q] += x[q];
      }
    }
  }
#pragma unroll
  for (int k = 0; k < kPtMaxK; ++k) {
    const int v = lane + 32 * k;
    if (v < hvec) {
#pragma unroll
      for (int q = 0; q < VE; ++q) pt_red[(size_t)warp * half + (size_t)v * VE + q] = acc[k][q];
    }
  }
  __syncthreads();
  const float invS = 1.f / wsum[b];
  for (int c = threadIdx.x; c < half; c += kPtWarps * 32) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kPtWarps; ++w) t += pt_red[(size_t)w * half + c];
    pt_red[(size_t)kPtWarps * half + c] = t * invS;                       // G / S
  }
  __syncthreads();
  float gs[kPtMaxK][8], pm[kPtMaxK][8];
#pragma unroll
  for (int k = 0; k < kPtMaxK; ++k) {
    const int v = lane + 32 * k;
#pragma unroll
    for (int q = 0; q < VE; ++q) {
      gs[k][q] = v < hvec ? pt_red[(size_t)kPtWarps * half + (size_t)v * VE + q] : 0.f;
      pm[k][q] = v < hvec ? pooled[(size_t)b * half + (size_t)v * VE + q] : 0.f;
    }
  }
  for (int n = warp; n < N; n += kPtWarps) {
    const float w = policy ? policy[(size_t)b * N + n] : 1.f;
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < kPtMaxK; ++k) {
      const int v = lane + 32 * k;
      if (v < hvec) {
        float o[8];
#pragma unroll
        for (int q = 0; q < VE; ++q) o[q] = w * gs[k][q];
        *reinterpret_cast<int4*>(db + (size_t)n * C + half + (size_t)v * VE) = PVec<T_>::pack(o);
        if (dpolicy) {
          float x[8];
          PVec<T_>::unpack(*reinterpret_cast<const int4*>(hb + (size_t)n * C + half + (size_t)v * VE), x);
#pragma unroll
          for (int q = 0; q < VE; ++q) dot = fmaf(x[q] - pm[k][q], gs[k][q], dot);
        }
      }
    }
    if (dpolicy) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
      if (lane == 0) dpolicy[(size_t)b * N + n] = dot;
    }
  }
}

}  // namespace d2s

using namespace d2s;

extern "C" int d2s_pool_act(const void* z, const float* policy, int dtype, int B, int N, int C, int act, void* local,
                            void* pooled, d2s_stream_t stream) {
  D2S_REQUIRE(z && pooled, D2S_ERR_ARG, "pool_act: null pointer");
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "pool_act: dtype %d unsupported", dtype);
  const int ve = dtype == D2S_BF16 ? 8 : 4;
  D2S_REQUIRE(B >= 0 && N >= 1 && C >= 2 * ve && C % (2 * ve) == 0 && C / ve <= kPoolThreads, D2S_ERR_ARG,
              "pool_act: bad shape B=%d N=%d C=%d (C must be a multiple of %d, at most %d)", B, N, C, 2 * ve, kPoolThreads * ve);
  D2S_REQUIRE(act >= D2S_ACT_NONE && act <= D2S_ACT_RELU, D2S_ERR_ARG, "pool_act: bad activation %d", act);
  D2S_REQUIRE(aligned16(z) && aligned16(local), D2S_ERR_ALIGN, "pool_act: z/local must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  const int groups = kPoolThreads / (local ? C / ve : C / ve / 2);
  const size_t smem = ((size_t)groups * (C / 2) + groups) * sizeof(float);
  if (dtype == D2S_BF16)
    pool_act_kernel<__nv_bfloat16><<<B, kPoolThreads, smem, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)z, policy, N, C, act, (__nv_bfloat16*)local, (__nv_bfloat16*)pooled, (long long)N * C);
  else
    pool_act_kernel<float><<<B, kPoolThreads, smem, (cudaStream_t)stream>>>((const float*)z, policy, N, C, act,
                                                                           (float*)local, (float*)pooled, (long long)N * C);
  count_launch();
  return check_launch("d2s_pool_act");
}

/* pooled only, over a row slice of a wider tensor: z points at the first pooled row of image 0, images are z_batch_stride elements
 * apart (e.g. x[:, 1:] of a (B, N + 1, C) tensor: z = x + C, z_batch_stride = (N + 1) * C).  bf16. */
extern "C" int d2s_pool_strided_bf16(const void* z, const float* policy, int B, int N, int C, long long z_batch_stride, int act,
                                     void* pooled, d2s_stream_t stream) {
  D2S_REQUIRE(z && pooled, D2S_ERR_ARG, "pool_strided: null pointer");
  D2S_REQUIRE(B >= 0 && N >= 1 && C >= 16 && C % 16 == 0 && C / 8 <= kPoolThreads, D2S_ERR_ARG, "pool_strided: bad shape B=%d N=%d C=%d", B, N, C);
  D2S_REQUIRE(z_batch_stride >= (long long)N * C && z_batch_stride % 8 == 0, D2S_ERR_ARG,
              "pool_strided: z_batch_stride=%lld must be a multiple of 8, at least N * C", z_batch_stride);
  D2S_REQUIRE(act >= D2S_ACT_NONE && act <= D2S_ACT_RELU, D2S_ERR_ARG, "pool_strided: bad activation %d", act);
  D2S_REQUIRE(aligned16(z), D2S_ERR_ALIGN, "pool_strided: z must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  const int groups = kPoolThreads / (C / 8 / 2);
  const size_t smem = ((size_t)groups * (C / 2) + groups) * sizeof(float);
  pool_act_kernel<__nv_bfloat16><<<B, kPoolThreads, smem, (cudaStream_t)stream>>>((const __nv_bfloat16*)z, policy, N, C, act, nullptr,
                                                                                 (__nv_bfloat16*)pooled, z_batch_stride);
  count_launch();
  return check_launch("d2s_pool_strided_bf16");
}

extern "C" int d2s_pool_concat_inplace(void* z, int dtype, int B, int N, int C, d2s_stream_t stream) {
  D2S_REQUIRE(z, D2S_ERR_ARG, "pool_concat_inplace: null pointer");
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "pool_concat_inplace: dtype %d unsupported", dtype);
  const int ve = dtype == D2S_BF16 ? 8 : 4;
  D2S_REQUIRE(B >= 0 && N >= 1 && C >= 2 * ve && C % (2 * ve) == 0 && C / ve / 2 <= kPoolThreads, D2S_ERR_ARG,
              "pool_concat_inplace: bad shape B=%d N=%d C=%d", B, N, C);
  D2S_REQUIRE(aligned16(z), D2S_ERR_ALIGN, "pool_concat_inplace: z must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  const int groups = kPoolThreads / (C / ve / 2);
  const size_t smem = ((size_t)groups + 1) * (C / 2) * sizeof(float);
  D2S_REQUIRE(smem <= 48 * 1024, D2S_ERR_ARG, "pool_concat_inplace: C=%d needs %zu B of shared memory", C, smem);
  if (dtype == D2S_BF16)
    pool_concat_inplace_kernel<__nv_bfloat16><<<B, kPoolThreads, smem, (cudaStream_t)stream>>>((__nv_bfloat16*)z, N, C, nullptr);
  else
    pool_concat_inplace_kernel<float><<<B, kPoolThreads, smem, (cudaStream_t)stream>>>((float*)z, N, C, nullptr);
  count_launch();
  return check_launch("d2s_pool_concat_inplace");
}

extern "C" int d2s_pool_concat_varlen_inplace(void* z, const int* n, int dtype, int B, int Nmax, int C, d2s_stream_t stream) {
  D2S_REQUIRE(z && n, D2S_ERR_ARG, "pool_concat_varlen_inplace: null pointer");
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "pool_concat_varlen_inplace: dtype %d unsupported", dtype);
  const int ve = dtype == D2S_BF16 ? 8 : 4;
  D2S_REQUIRE(B >= 0 && Nmax >= 1 && C >= 2 * ve && C % (2 * ve) == 0 && C / ve / 2 <= kPoolThreads, D2S_ERR_ARG,
              "pool_concat_varlen_inplace: bad shape B=%d Nmax=%d C=%d", B, Nmax, C);
  D2S_REQUIRE(aligned16(z), D2S_ERR_ALIGN, "pool_concat_varlen_inplace: z must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  const int groups = kPoolThreads / (C / ve / 2);
  const size_t smem = ((size_t)groups + 1) * (C / 2) * sizeof(float);
  D2S_REQUIRE(smem <= 48 * 1024, D2S_ERR_ARG, "pool_concat_varlen_inplace: C=%d needs %zu B of shared memory", C, smem);
  if (dtype == D2S_BF16)
    pool_concat_inplace_kernel<__nv_bfloat16, true><<<B, kPoolThreads, smem, (cudaStream_t)stream>>>((__nv_bfloat16*)z, Nmax, C, n);
  else
    pool_concat_inplace_kernel<float, true><<<B, kPoolThreads, smem, (cudaStream_t)stream>>>((float*)z, Nmax, C, n);
  count_launch();
  return check_launch("d2s_pool_concat_varlen_inplace");
}

extern "C" int d2s_bias_act(void* u, const void* bias, int dtype, long long rows, int N, int C, int act, d2s_stream_t stream) {
  D2S_REQUIRE(u, D2S_ERR_ARG, "bias_act: null pointer");
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "bias_act: dtype %d unsupported", dtype);
  const int ve = dtype == D2S_BF16 ? 8 : 4;
  D2S_REQUIRE(rows >= 0 && N >= 0 && C >= ve && C % ve == 0, D2S_ERR_ARG, "bias_act: bad shape rows=%lld N=%d C=%d", rows, N, C);
  D2S_REQUIRE(act >= D2S_ACT_NONE && act <= D2S_ACT_RELU, D2S_ERR_ARG, "bias_act: bad activation %d", act);
  D2S_REQUIRE(aligned16(u) && (!bias || aligned16(bias)), D2S_ERR_ALIGN, "bias_act: u/bias must be 16-byte aligned");
  if (rows == 0) return D2S_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (bias == nullptr) {
    const long long total = rows * (C / ve);
    long long blocks = (total + 511) / 512;
    if (blocks > 16LL * kNumSMs) blocks = 16LL * kNumSMs;
    if (dtype == D2S_BF16) act_flat_kernel<__nv_bfloat16><<<(unsigned)blocks, 256, 0, st>>>((__nv_bfloat16*)u, total, act);
    else                   act_flat_kernel<float><<<(unsigned)blocks, 256, 0, st>>>((float*)u, total, act);
  } else {
    const long long nblk = (rows + kBiasRows - 1) / kBiasRows;
    D2S_REQUIRE(nblk <= 0x7fffffffLL, D2S_ERR_ARG, "bias_act: too many rows %lld", rows);
    const unsigned grid = (unsigned)nblk;
    if (dtype == D2S_BF16)
      bias_act_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((__nv_bfloat16*)u, (const __nv_bfloat16*)bias, rows, N, C, act);
    else
      bias_act_kernel<float><<<grid, 256, 0, st>>>((float*)u, (const float*)bias, rows, N, C, act);
  }
  count_launch();
  return check_launch("d2s_bias_act");
}

static int pool_concat_check(const char* what, int dtype, int B, int N, int C) {
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "%s: dtype %d unsupported", what, dtype);
  const int ve = dtype == D2S_BF16 ? 8 : 4;
  D2S_REQUIRE(B >= 0 && N >= 1 && C >= 2 * ve && C % (2 * ve) == 0 && C / 2 / ve <= 32 * kPtMaxK, D2S_ERR_ARG,
              "%s: bad shape B=%d N=%d C=%d (C/2 a multiple of %d, at most %d)", what, B, N, C, ve, 32 * kPtMaxK * ve);
  return D2S_OK;
}

extern "C" int d2s_pool_concat_fwd(const void* h, const float* policy, int dtype, int B, int N, int C, void* out, float* pooled,
                                   float* wsum, d2s_stream_t stream) {
  D2S_REQUIRE(h && out && pooled && wsum, D2S_ERR_ARG, "pool_concat_fwd: null pointer");
  int rc = pool_concat_check("pool_concat_fwd", dtype, B, N, C);
  if (rc) return rc;
  D2S_REQUIRE(aligned16(h) && aligned16(out), D2S_ERR_ALIGN, "pool_concat_fwd: h/out must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  const size_t smem = ((size_t)kPtWarps + 1) * (C / 2) * sizeof(float);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == D2S_BF16)
    pool_concat_fwd_kernel<__nv_bfloat16><<<B, kPtWarps * 32, smem, st>>>((const __nv_bfloat16*)h, policy, N, C, (__nv_bfloat16*)out, pooled, wsum);
  else
    pool_concat_fwd_kernel<float><<<B, kPtWarps * 32, smem, st>>>((const float*)h, policy, N, C, (float*)out, pooled, wsum);
  count_launch();
  return check_launch("d2s_pool_concat_fwd");
}

extern "C" int d2s_pool_concat_bwd(const void* dout, const void* h, const float* policy, const float* pooled, const float* wsum,
                                   int dtype, int B, int N, int C, void* dh, float* dpolicy, d2s_stream_t stream) {
  D2S_REQUIRE(dout && h && pooled && wsum && dh, D2S_ERR_ARG, "pool_concat_bwd: null pointer");
  D2S_REQUIRE(!dpolicy || policy, D2S_ERR_ARG, "pool_concat_bwd: dpolicy without a policy");
  int rc = pool_concat_check("pool_concat_bwd", dtype, B, N, C);
  if (rc) return rc;
  D2S_REQUIRE(aligned16(dout) && aligned16(h) && aligned16(dh), D2S_ERR_ALIGN, "pool_concat_bwd: dout/h/dh must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  const size_t smem = ((size_t)kPtWarps + 1) * (C / 2) * sizeof(float);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == D2S_BF16)
    pool_concat_bwd_kernel<__nv_bfloat16><<<B, kPtWarps * 32, smem, st>>>((const __nv_bfloat16*)dout, (const __nv_bfloat16*)h, policy, pooled,
                                                                         wsum, N, C, (__nv_bfloat16*)dh, dpolicy);
  else
    pool_concat_bwd_kernel<float><<<B, kPtWarps * 32, smem, st>>>((const float*)dout, (const float*)h, policy, pooled, wsum, N, C,
                                                                  (float*)dh, dpolicy);
  count_launch();
  return check_launch("d2s_pool_concat_bwd");
}
