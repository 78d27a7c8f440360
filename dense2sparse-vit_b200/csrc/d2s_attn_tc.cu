// Entry point of the tcgen05 attention forward (d2s_attn_policy_fwd); the kernel is in d2s_attn_tc.cuh.  Its variable-length
// instantiations live in d2s_attn_varlen.cu: compiled in this translation unit they changed the code generated for the dense ones.
#include "d2s_attn_tc.cuh"


using namespace d2s;

#ifdef D2S_ATTN_TRACE_BUILD
extern "C" int d2s_debug_attn_trace(long long* host_out, int n_ctas) {   // profiling builds only; not part of include/d2s.h
  cudaDeviceSynchronize();
  return (int)cudaMemcpyFromSymbol(host_out, d2s_tc_trace_buf, (size_t)n_ctas * 16 * sizeof(long long));
}
#endif

extern "C" int d2s_attn_policy_fwd(const void* qkv, const float* policy, int dtype, int B, int T, int H, int hd,
                                   float scale, float eps, void* out, float* cls_row, float* stats, d2s_stream_t stream_) {
  D2S_REQUIRE(qkv && out, D2S_ERR_ARG, "attn_policy_fwd: null pointer");
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "attn_policy_fwd: dtype %d unsupported", dtype);
  D2S_REQUIRE(B >= 0 && T >= 1 && H >= 1 && hd >= 1, D2S_ERR_ARG, "attn_policy_fwd: bad shape B=%d T=%d H=%d hd=%d", B, T, H, hd);
  D2S_REQUIRE((long long)B * H <= (1LL << 30), D2S_ERR_ARG, "attn_policy_fwd: B*H=%lld too large", (long long)B * H);
  D2S_REQUIRE(aligned16(qkv) && aligned16(out) && aligned16(stats), D2S_ERR_ALIGN,
              "attn_policy_fwd: qkv/out/stats must be 16-byte aligned");
  D2S_REQUIRE(scale > 0.0f, D2S_ERR_ARG, "attn_policy_fwd: scale must be positive (got %g)", (double)scale);
  cudaStream_t stream = (cudaStream_t)stream_;
  if (dtype == D2S_F32) {
    D2S_REQUIRE(stats == nullptr, D2S_ERR_ARG, "attn_policy_fwd: row statistics are written by the bf16 tcgen05 kernel only");
    D2S_REQUIRE((long long)B * H <= 65535, D2S_ERR_ARG, "attn_policy_fwd(simt): B*H=%lld exceeds 65535", (long long)B * H);
    if (B == 0) return D2S_OK;
    return attn_simt_dispatch(qkv, policy, B, T, H, hd, scale, eps, out, cls_row, stream);
  }
  D2S_REQUIRE(hd == kTcHD, D2S_ERR_ARG, "attn_policy_fwd(bf16): head dim %d unsupported by the tcgen05 kernel (64 only)", hd);
  D2S_REQUIRE(T <= 256, D2S_ERR_ARG, "attn_policy_fwd(bf16): T=%d exceeds 256", T);
  if (B == 0) return D2S_OK;
  const int Tkp = ceil_div(T, 16) * 16;
  CUtensorMap map_a, map_b;
  int rc = encode_qkv_maps(qkv, B, T, H, Tkp, map_a, map_b);
  if (rc) return rc;
  const int units = B * H;
  if (T <= kTileRows) {
    return policy ? launch_tc<1, true, 4>(map_a, map_b, policy, units, T, H, Tkp, scale, eps, out, cls_row, stats, qkv, stream)
                  : launch_tc<1, false, 4>(map_a, map_b, policy, units, T, H, Tkp, scale, eps, out, cls_row, stats, qkv, stream);
  }
  return policy ? launch_tc<2, true, 8>(map_a, map_b, policy, units, T, H, Tkp, scale, eps, out, cls_row, stats, qkv, stream)
                : launch_tc<2, false, 8>(map_a, map_b, policy, units, T, H, Tkp, scale, eps, out, cls_row, stats, qkv, stream);
}
