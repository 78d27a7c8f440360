// Residual add + LayerNorm in one pass over the token matrix (inference path of Block.forward,
// vit_models/dynamic_vit.py:263-283 / default_dynamic_vit.py:234-237, and of the predictors' leading LayerNorm,
// dynamic_vit.py:409 / default_dynamic_vit.py:308):
//
//     s = x + y            (rounded to the tensor dtype, exactly like the reference's separate add)
//     h = LayerNorm(s) * gamma + beta     (statistics in fp32, two-pass over registers)
//
// HBM-bound byte movement: per token row 2*e*D bytes in (x, y) and 2*e*D out (s, h); the reference's eager path
// moves 5*e*D (add: 2 in 1 out, LayerNorm: 1 in 1 out) in two launches, and torch's bf16 LayerNorm kernel runs at a
// fifth of HBM speed at D=384 (profiles/README.md, r01a).  One half-warp owns a row: 16 lanes x 16-byte vectors
// cover D=384 bf16 in exactly 3 vectors per lane; reductions are 4 xor-shuffles inside the half-warp.
#include "d2s_common.cuh"

namespace d2s {

constexpr int kLnThreads = 256;

template <typename T_> struct LnVec;
template <> struct LnVec<__nv_bfloat16> {
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
template <> struct LnVec<float> {
  static constexpr int kElems = 4;
  __device__ static void unpack(const int4& r, float (&v)[8]) {
    v[0] = __int_as_float(r.x); v[1] = __int_as_float(r.y); v[2] = __int_as_float(r.z); v[3] = __int_as_float(r.w);
  }
  __device__ static int4 pack(const float (&v)[8]) {
    return make_int4(__float_as_int(v[0]), __float_as_int(v[1]), __float_as_int(v[2]), __float_as_int(v[3]));
  }
  __device__ static float round(float f) { return f; }
};

template <int kLPR>
__device__ __forceinline__ float row_lanes_sum(float v) {
#pragma unroll
  for (int o = kLPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// kLPR lanes per row (16: two rows per warp; 32 for wide rows -- at 12 vectors per lane the 1536-wide predictor LayerNorm ran at
// 2.6 TB/s), kVPL 16-byte vectors per lane (D <= kLPR * kVPL * elems-per-vector)
// kVar: variable-length gather (d2s_gather_layernorm_varlen): output token t >= 1 of image b is a pad row when t - 1 >= cnt[b]; it
// is processed as a zero row (its index is not read) and written as zeros, out_norm included.
template <typename T_, int kVPL, int kLPR, bool kVar = false>
__global__ void __launch_bounds__(kLnThreads)
add_layernorm_kernel(const T_* __restrict__ x, const T_* __restrict__ y, const T_* __restrict__ gamma,
                     const T_* __restrict__ beta, long long rows, int T, int D, long long x_stride_b, long long x_stride_t,
                     float eps, int norm_row0, T_* __restrict__ out_sum, T_* __restrict__ out_norm,
                     const int64_t* __restrict__ gather_idx, const T_* __restrict__ cls_row, float2* __restrict__ stats,
                     const int* __restrict__ cnt) {
  constexpr int VE = LnVec<T_>::kElems;
  const int sub = threadIdx.x & (kLPR - 1);
  const long long row = (long long)blockIdx.x * (kLnThreads / kLPR) + threadIdx.x / kLPR;
  const int nvec = D / VE;
  const long long b = row < rows ? row / T : 0;
  const int t = row < rows ? (int)(row - b * T) : 0;
  const bool pad = kVar && row < rows && t > 0 && t - 1 >= cnt[b];
  const bool row_ok = row < rows && !pad;   // a row whose input is read
  // gather mode (d2s_gather_layernorm): output token 0 is the CLS row, token t >= 1 is input token idx[b, t-1] + 1
  const long long src_t = (gather_idx && row_ok && t > 0) ? gather_idx[b * (T - 1) + (t - 1)] + 1 : (long long)t;
  // assemble mode (d2s_assemble_layernorm, cls_row != NULL): token 0 is the class token, token t >= 1 is patch t-1 of x, and
  // y is the position embedding, one row per TOKEN shared by all images
  const T_* xr = (cls_row && t == 0) ? cls_row : x + b * x_stride_b + (src_t - (cls_row ? 1 : 0)) * x_stride_t;
  const T_* yr = y ? y + (cls_row ? (long long)t : row) * D : nullptr;

  float v[kVPL][8];
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < kVPL; ++k) {
    const int vi = sub + kLPR * k;
    if (row_ok && vi < nvec) {
      const int4 rx = *reinterpret_cast<const int4*>(xr + (size_t)vi * VE);
      LnVec<T_>::unpack(rx, v[k]);
      if (yr) {
        float w[8];
        const int4 ry = ld_stream16(yr + (size_t)vi * VE);  // the branch output is dead after this read
        LnVec<T_>::unpack(ry, w);
#pragma unroll
        for (int q = 0; q < VE; ++q) v[k][q] = LnVec<T_>::round(v[k][q] + w[q]);
      }
#pragma unroll
      for (int q = 0; q < VE; ++q) sum += v[k][q];
    } else {
#pragma unroll
      for (int q = 0; q < VE; ++q) v[k][q] = 0.f;
    }
  }
  if (out_sum && (row_ok || pad)) {
#pragma unroll
    for (int k = 0; k < kVPL; ++k) {
      const int vi = sub + kLPR * k;
      if (vi < nvec) *reinterpret_cast<int4*>(out_sum + row * D + (size_t)vi * VE) = LnVec<T_>::pack(v[k]);
    }
  }
  const float mean = row_lanes_sum<kLPR>(sum) / (float)D;
  float var = 0.f;
#pragma unroll
  for (int k = 0; k < kVPL; ++k) {
    const int vi = sub + kLPR * k;
    if (vi < nvec) {
#pragma unroll
      for (int q = 0; q < VE; ++q) {
        const float d = v[k][q] - mean;
        var = fmaf(d, d, var);
      }
    }
  }
  const float rstd = rsqrtf(row_lanes_sum<kLPR>(var) / (float)D + eps);
  // per-row (mean, rstd) for a consumer that applies the LayerNorm itself (the qkv GEMM on its resident input rows); out_norm may
  // then be NULL.  For bf16 both forms use h = fma(fma(x, rstd, -mean * rstd), gamma, beta), so they give the same bits.
  if (stats != nullptr && (row_ok || pad) && sub == 0) stats[row] = make_float2(mean, rstd);
  if (!(row_ok || pad) || t < norm_row0 || out_norm == nullptr) return;
  const float shift = -mean * rstd;
  T_* hr = out_norm + (b * (T - norm_row0) + (t - norm_row0)) * (long long)D;
#pragma unroll
  for (int k = 0; k < kVPL; ++k) {
    const int vi = sub + kLPR * k;
    if (vi < nvec) {
      float g[8], bt[8], o[8];
      LnVec<T_>::unpack(*reinterpret_cast<const int4*>(gamma + (size_t)vi * VE), g);
      LnVec<T_>::unpack(*reinterpret_cast<const int4*>(beta + (size_t)vi * VE), bt);
#pragma unroll
      for (int q = 0; q < VE; ++q)     // bf16: the form the GEMM kernels use (same bits as the on-the-fly norm); fp32: the more accurate one
        o[q] = pad ? 0.f : sizeof(T_) == 2 ? fmaf(fmaf(v[k][q], rstd, shift), g[q], bt[q]) : fmaf((v[k][q] - mean) * rstd, g[q], bt[q]);
      *reinterpret_cast<int4*>(hr + (size_t)vi * VE) = LnVec<T_>::pack(o);
    }
  }
}

// LayerNorm applied from GIVEN per-row statistics (bf16): out[r] = bf16(fma(fma(x[r], rstd_r, -mean_r * rstd_r), gamma, beta)) -- the
// arithmetic the GEMM kernels use when they normalise their input tiles themselves, for the few rows another consumer needs
// materialised (the CLS rows in front of the CLS-only last MLP).  One warp per row.
__global__ void apply_ln_stats_kernel(const __nv_bfloat16* __restrict__ x, const float2* __restrict__ stats,
                                      const __nv_bfloat16* __restrict__ gamma, const __nv_bfloat16* __restrict__ beta, int rows, int D,
                                      long long x_row_stride, long long stat_row_stride, __nv_bfloat16* __restrict__ out) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float2 st = stats[(long long)row * stat_row_stride];
  const float shift = -st.x * st.y;
  const __nv_bfloat16* xr = x + (long long)row * x_row_stride;
  for (int c = lane; c < D; c += 32)
    out[(long long)row * D + c] =
        __float2bfloat16_rn(fmaf(fmaf(__bfloat162float(xr[c]), st.y, shift), __bfloat162float(gamma[c]), __bfloat162float(beta[c])));
}

template <typename T_, bool kVar = false>
static int launch_ln(const void* x, const void* y, const void* gamma, const void* beta, int B, int T, int D,
                     long long sb, long long st, float eps, int norm_row0, void* out_sum, void* out_norm, cudaStream_t stream,
                     const int64_t* gather_idx = nullptr, const void* cls_row = nullptr, float* stats = nullptr,
                     const int* cnt = nullptr) {
  constexpr int VE = LnVec<T_>::kElems;
  const long long rows = (long long)B * T;
  const int nvec = D / VE;
  const int vpl = ceil_div(nvec, 16);
#define D2S_LN_LAUNCH(V, L)                                                                                            \
  add_layernorm_kernel<T_, V, L, kVar><<<(unsigned)((rows + kLnThreads / L - 1) / (kLnThreads / L)), kLnThreads, 0, stream>>>(  \
      (const T_*)x, (const T_*)y, (const T_*)gamma, (const T_*)beta, rows, T, D, sb, st, eps, norm_row0, (T_*)out_sum,     \
      (T_*)out_norm, gather_idx, (const T_*)cls_row, reinterpret_cast<float2*>(stats), cnt)
  if (vpl <= 2) D2S_LN_LAUNCH(2, 16);
  else if (vpl <= 3) D2S_LN_LAUNCH(3, 16);
  else if (vpl <= 6) D2S_LN_LAUNCH(3, 32);
  else D2S_LN_LAUNCH(6, 32);
#undef D2S_LN_LAUNCH
  count_launch();
  return check_launch(kVar ? "d2s_gather_layernorm_varlen" : "d2s_add_layernorm");
}

}  // namespace d2s

using namespace d2s;

extern "C" int d2s_add_layernorm(const void* x, const void* y, const void* gamma, const void* beta, int dtype, int B, int T,
                                 int D, long long x_stride_b, long long x_stride_t, float eps, int norm_row0,
                                 void* out_sum, void* out_norm, d2s_stream_t stream) {
  D2S_REQUIRE(x && gamma && beta && out_norm, D2S_ERR_ARG, "add_layernorm: null pointer");
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "add_layernorm: dtype %d unsupported", dtype);
  D2S_REQUIRE(B >= 0 && T >= 1 && D >= 1, D2S_ERR_ARG, "add_layernorm: bad shape B=%d T=%d D=%d", B, T, D);
  const int ve = dtype == D2S_BF16 ? 8 : 4;
  D2S_REQUIRE(D % ve == 0 && D / ve <= 16 * 12, D2S_ERR_ARG, "add_layernorm: D=%d must be a multiple of %d and at most %d", D,
              ve, 16 * 12 * ve);
  D2S_REQUIRE(norm_row0 >= 0 && norm_row0 < T, D2S_ERR_ARG, "add_layernorm: norm_row0=%d outside [0,T=%d)", norm_row0, T);
  D2S_REQUIRE(x_stride_t >= D && x_stride_b >= 0 && x_stride_t % ve == 0 && x_stride_b % ve == 0, D2S_ERR_ARG,
              "add_layernorm: strides (%lld, %lld) must be multiples of %d elements with rows >= D apart", x_stride_b,
              x_stride_t, ve);
  D2S_REQUIRE(aligned16(x) && aligned16(gamma) && aligned16(beta) && aligned16(out_norm) && (!y || aligned16(y)) &&
                  (!out_sum || aligned16(out_sum)),
              D2S_ERR_ALIGN, "add_layernorm: pointers must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  return dtype == D2S_BF16
             ? launch_ln<__nv_bfloat16>(x, y, gamma, beta, B, T, D, x_stride_b, x_stride_t, eps, norm_row0, out_sum, out_norm,
                                        (cudaStream_t)stream)
             : launch_ln<float>(x, y, gamma, beta, B, T, D, x_stride_b, x_stride_t, eps, norm_row0, out_sum, out_norm,
                                (cudaStream_t)stream);
}

/* Kept-token gather fused with the LayerNorm that follows it (default_dynamic_vit.py:464-468 + Block.forward's norm1,
 * dynamic_vit.py:907-912 + :263): out_sum (B,K+1,D) = [CLS, x[idx+1]], out_norm = LayerNorm(out_sum) * gamma + beta. */
extern "C" int d2s_gather_layernorm(const void* x, const int64_t* idx, const void* gamma, const void* beta, int dtype, int B,
                                    int T_in, int D, int K, float eps, void* out_sum, void* out_norm, d2s_stream_t stream) {
  D2S_REQUIRE(x && (idx || K == 0) && gamma && beta && out_sum && out_norm, D2S_ERR_ARG, "gather_layernorm: null pointer");
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "gather_layernorm: dtype %d unsupported", dtype);
  D2S_REQUIRE(B >= 0 && T_in >= 1 && D >= 1 && K >= 0 && K <= T_in - 1, D2S_ERR_ARG,
              "gather_layernorm: bad shape B=%d T_in=%d D=%d K=%d", B, T_in, D, K);
  const int ve = dtype == D2S_BF16 ? 8 : 4;
  D2S_REQUIRE(D % ve == 0 && D / ve <= 16 * 12, D2S_ERR_ARG, "gather_layernorm: D=%d must be a multiple of %d and at most %d", D,
              ve, 16 * 12 * ve);
  D2S_REQUIRE(aligned16(x) && aligned16(gamma) && aligned16(beta) && aligned16(out_sum) && aligned16(out_norm), D2S_ERR_ALIGN,
              "gather_layernorm: pointers must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  const long long sb = (long long)T_in * D, st = D;
  return dtype == D2S_BF16
             ? launch_ln<__nv_bfloat16>(x, nullptr, gamma, beta, B, K + 1, D, sb, st, eps, 0, out_sum, out_norm, (cudaStream_t)stream, K ? idx : nullptr)
             : launch_ln<float>(x, nullptr, gamma, beta, B, K + 1, D, sb, st, eps, 0, out_sum, out_norm, (cudaStream_t)stream,
                                K ? idx : nullptr);
}

/* Token assembly fused with the first block's norm1 (dynamic_vit.py:820-823 + Block.forward :263): out_sum (B,N+1,D) =
 * cat(cls, patches) + pos, out_norm = LayerNorm(out_sum) * gamma + beta.  patches (B,N,D), cls (D), pos (N+1,D). */
extern "C" int d2s_assemble_layernorm(const void* patches, const void* cls, const void* pos, const void* gamma, const void* beta,
                                      int dtype, int B, int N, int D, float eps, void* out_sum, void* out_norm,
                                      d2s_stream_t stream) {
  D2S_REQUIRE(patches && cls && pos && gamma && beta && out_sum && out_norm, D2S_ERR_ARG, "assemble_layernorm: null pointer");
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "assemble_layernorm: dtype %d unsupported", dtype);
  D2S_REQUIRE(B >= 0 && N >= 1 && D >= 1, D2S_ERR_ARG, "assemble_layernorm: bad shape B=%d N=%d D=%d", B, N, D);
  const int ve = dtype == D2S_BF16 ? 8 : 4;
  D2S_REQUIRE(D % ve == 0 && D / ve <= 16 * 12, D2S_ERR_ARG, "assemble_layernorm: D=%d must be a multiple of %d and at most %d", D,
              ve, 16 * 12 * ve);
  D2S_REQUIRE(aligned16(patches) && aligned16(cls) && aligned16(pos) && aligned16(gamma) && aligned16(beta) && aligned16(out_sum) &&
                  aligned16(out_norm),
              D2S_ERR_ALIGN, "assemble_layernorm: pointers must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  const long long sb = (long long)N * D, st = D;
  return dtype == D2S_BF16 ? launch_ln<__nv_bfloat16>(patches, pos, gamma, beta, B, N + 1, D, sb, st, eps, 0, out_sum, out_norm,
                                                      (cudaStream_t)stream, nullptr, cls)
                           : launch_ln<float>(patches, pos, gamma, beta, B, N + 1, D, sb, st, eps, 0, out_sum, out_norm,
                                              (cudaStream_t)stream, nullptr, cls);
}

/* The same two with per-row (mean, rstd) of out_sum instead of the normalised output (bf16): the consumer -- the first / next
 * block's qkv projection, d2s_linear_lnin_act_pair_bf16 -- applies norm1 to its resident input rows itself, so LayerNorm(out_sum)
 * is never written or read.  stats (B*(K+1), 2) / (B*(N+1), 2) f32. */
extern "C" int d2s_gather_layernorm_stats(const void* x, const int64_t* idx, int B, int T_in, int D, int K, float eps, void* out_sum,
                                          float* stats, d2s_stream_t stream) {
  D2S_REQUIRE(x && (idx || K == 0) && out_sum && stats, D2S_ERR_ARG, "gather_layernorm_stats: null pointer");
  D2S_REQUIRE(B >= 0 && T_in >= 1 && D >= 8 && K >= 0 && K <= T_in - 1 && D % 8 == 0 && D / 8 <= 16 * 12, D2S_ERR_ARG,
              "gather_layernorm_stats: bad shape B=%d T_in=%d D=%d K=%d", B, T_in, D, K);
  D2S_REQUIRE(aligned16(x) && aligned16(out_sum) && (reinterpret_cast<uintptr_t>(stats) & 7u) == 0, D2S_ERR_ALIGN,
              "gather_layernorm_stats: x / out_sum must be 16-byte aligned, stats 8-byte aligned");
  if (B == 0) return D2S_OK;
  return launch_ln<__nv_bfloat16>(x, nullptr, x, x, B, K + 1, D, (long long)T_in * D, D, eps, 0, out_sum, nullptr, (cudaStream_t)stream,
                                  K ? idx : nullptr, nullptr, stats);
}

/* Variable-length forms of the two gathers above (threshold inference): idx (B,Kmax) holds image b's count[b] kept spatial indices
 * followed by padding (never read); output rows 1 + count[b] .. Kmax of out_sum / out_norm are zeros, stats of those rows are the
 * (mean, rstd) of a zero row. */
extern "C" int d2s_gather_layernorm_varlen(const void* x, const int64_t* idx, const int* count, const void* gamma, const void* beta,
                                           int dtype, int B, int T_in, int D, int Kmax, float eps, void* out_sum, void* out_norm,
                                           d2s_stream_t stream) {
  D2S_REQUIRE(x && (idx || Kmax == 0) && count && gamma && beta && out_sum && out_norm, D2S_ERR_ARG, "gather_layernorm_varlen: null pointer");
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "gather_layernorm_varlen: dtype %d unsupported", dtype);
  D2S_REQUIRE(B >= 0 && T_in >= 1 && D >= 1 && Kmax >= 0 && Kmax <= T_in - 1, D2S_ERR_ARG,
              "gather_layernorm_varlen: bad shape B=%d T_in=%d D=%d Kmax=%d", B, T_in, D, Kmax);
  const int ve = dtype == D2S_BF16 ? 8 : 4;
  D2S_REQUIRE(D % ve == 0 && D / ve <= 16 * 12, D2S_ERR_ARG, "gather_layernorm_varlen: D=%d must be a multiple of %d and at most %d",
              D, ve, 16 * 12 * ve);
  D2S_REQUIRE(aligned16(x) && aligned16(gamma) && aligned16(beta) && aligned16(out_sum) && aligned16(out_norm), D2S_ERR_ALIGN,
              "gather_layernorm_varlen: pointers must be 16-byte aligned");
  if (B == 0) return D2S_OK;
  const long long sb = (long long)T_in * D, st = D;
  return dtype == D2S_BF16
             ? launch_ln<__nv_bfloat16, true>(x, nullptr, gamma, beta, B, Kmax + 1, D, sb, st, eps, 0, out_sum, out_norm,
                                              (cudaStream_t)stream, Kmax ? idx : nullptr, nullptr, nullptr, count)
             : launch_ln<float, true>(x, nullptr, gamma, beta, B, Kmax + 1, D, sb, st, eps, 0, out_sum, out_norm, (cudaStream_t)stream,
                                      Kmax ? idx : nullptr, nullptr, nullptr, count);
}

extern "C" int d2s_gather_layernorm_stats_varlen(const void* x, const int64_t* idx, const int* count, int B, int T_in, int D, int Kmax,
                                                 float eps, void* out_sum, float* stats, d2s_stream_t stream) {
  D2S_REQUIRE(x && (idx || Kmax == 0) && count && out_sum && stats, D2S_ERR_ARG, "gather_layernorm_stats_varlen: null pointer");
  D2S_REQUIRE(B >= 0 && T_in >= 1 && D >= 8 && Kmax >= 0 && Kmax <= T_in - 1 && D % 8 == 0 && D / 8 <= 16 * 12, D2S_ERR_ARG,
              "gather_layernorm_stats_varlen: bad shape B=%d T_in=%d D=%d Kmax=%d", B, T_in, D, Kmax);
  D2S_REQUIRE(aligned16(x) && aligned16(out_sum) && (reinterpret_cast<uintptr_t>(stats) & 7u) == 0, D2S_ERR_ALIGN,
              "gather_layernorm_stats_varlen: x / out_sum must be 16-byte aligned, stats 8-byte aligned");
  if (B == 0) return D2S_OK;
  return launch_ln<__nv_bfloat16, true>(x, nullptr, x, x, B, Kmax + 1, D, (long long)T_in * D, D, eps, 0, out_sum, nullptr,
                                        (cudaStream_t)stream, Kmax ? idx : nullptr, nullptr, stats, count);
}

extern "C" int d2s_assemble_layernorm_stats(const void* patches, const void* cls, const void* pos, int B, int N, int D, float eps,
                                            void* out_sum, float* stats, d2s_stream_t stream) {
  D2S_REQUIRE(patches && cls && pos && out_sum && stats, D2S_ERR_ARG, "assemble_layernorm_stats: null pointer");
  D2S_REQUIRE(B >= 0 && N >= 1 && D >= 8 && D % 8 == 0 && D / 8 <= 16 * 12, D2S_ERR_ARG, "assemble_layernorm_stats: bad shape B=%d N=%d D=%d",
              B, N, D);
  D2S_REQUIRE(aligned16(patches) && aligned16(cls) && aligned16(pos) && aligned16(out_sum) && (reinterpret_cast<uintptr_t>(stats) & 7u) == 0,
              D2S_ERR_ALIGN, "assemble_layernorm_stats: pointers must be 16-byte aligned, stats 8-byte aligned");
  if (B == 0) return D2S_OK;
  return launch_ln<__nv_bfloat16>(patches, pos, patches, patches, B, N + 1, D, (long long)N * D, D, eps, 0, out_sum, nullptr,
                                  (cudaStream_t)stream, nullptr, cls, stats);
}

/* out (rows, D) = LayerNorm of rows of x taken from GIVEN statistics: row r of x at x + r * x_row_stride elements, its (mean, rstd)
 * at stats + 2 * r * stat_row_stride floats (bf16; same arithmetic as the GEMM kernels' on-the-fly normalisation). */
extern "C" int d2s_apply_layernorm_stats_bf16(const void* x, const float* stats, const void* gamma, const void* beta, int rows, int D,
                                              long long x_row_stride, long long stat_row_stride, void* out, d2s_stream_t stream) {
  D2S_REQUIRE(x && stats && gamma && beta && out, D2S_ERR_ARG, "apply_layernorm_stats: null pointer");
  D2S_REQUIRE(rows >= 0 && D >= 1 && x_row_stride >= D && stat_row_stride >= 1, D2S_ERR_ARG,
              "apply_layernorm_stats: bad shape rows=%d D=%d strides (%lld, %lld)", rows, D, x_row_stride, stat_row_stride);
  if (rows == 0) return D2S_OK;
  apply_ln_stats_kernel<<<(rows + 7) / 8, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, reinterpret_cast<const float2*>(stats),
                                                                         (const __nv_bfloat16*)gamma, (const __nv_bfloat16*)beta, rows, D,
                                                                         x_row_stride, stat_row_stride, (__nv_bfloat16*)out);
  count_launch();
  return check_launch("d2s_apply_layernorm_stats_bf16");
}
