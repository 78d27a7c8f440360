// Kernel family (4), CUDA-core part:
//   * softmax_with_policy forward/backward over a materialised (B,H,T,T) score tensor -- the drop-in for
//     Attention.softmax_with_policy (vit_models/dynamic_vit.py:195-214), one pass instead of the reference's
//     ~11 elementwise passes; used by the patched reference and by the training inputs the tcgen05
//     attention pairs do not take (fp32, head dim != 64);
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
