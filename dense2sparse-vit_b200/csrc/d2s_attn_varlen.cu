// Variable-length entry point of the attention forward (d2s_attn_varlen_fwd): the kernels of d2s_attn_tc.cuh with kVar = true, in
// a translation unit of their own so that the dense instantiations in d2s_attn_tc.cu compile exactly as before.
#undef D2S_ATTN_TRACE_BUILD   // the clock64 phase traces instrument the dense kernels only
#include "d2s_attn_tc.cuh"

using namespace d2s;

/* Variable-length form (threshold inference, dynamic_vit.py:935-960 batched): qkv (B,Tmax,3,H,hd), image b valid in its first
 * lens[b] rows; out (B,Tmax,H*hd) and cls_row (B,H,Tmax) zero past lens[b].  No policy, no row statistics. */
extern "C" int d2s_attn_varlen_fwd(const void* qkv, const int* lens, int dtype, int B, int Tmax, int H, int hd, float scale,
                                   void* out, float* cls_row, d2s_stream_t stream_) {
  D2S_REQUIRE(qkv && lens && out, D2S_ERR_ARG, "attn_varlen_fwd: null pointer");
  D2S_REQUIRE(dtype == D2S_F32 || dtype == D2S_BF16, D2S_ERR_ARG, "attn_varlen_fwd: dtype %d unsupported", dtype);
  D2S_REQUIRE(B >= 0 && Tmax >= 1 && Tmax <= 256 && H >= 1 && hd >= 1, D2S_ERR_ARG,
              "attn_varlen_fwd: bad shape B=%d Tmax=%d H=%d hd=%d (Tmax <= 256)", B, Tmax, H, hd);
  D2S_REQUIRE((long long)B * H <= (1LL << 30), D2S_ERR_ARG, "attn_varlen_fwd: B*H=%lld too large", (long long)B * H);
  D2S_REQUIRE(aligned16(qkv) && aligned16(out), D2S_ERR_ALIGN, "attn_varlen_fwd: qkv/out must be 16-byte aligned");
  D2S_REQUIRE(scale > 0.0f, D2S_ERR_ARG, "attn_varlen_fwd: scale must be positive (got %g)", (double)scale);
  cudaStream_t stream = (cudaStream_t)stream_;
  if (dtype == D2S_F32) {
    D2S_REQUIRE((long long)B * H <= 65535, D2S_ERR_ARG, "attn_varlen_fwd(simt): B*H=%lld exceeds 65535", (long long)B * H);
    if (B == 0) return D2S_OK;
    return attn_simt_dispatch(qkv, nullptr, B, Tmax, H, hd, scale, 0.0f, out, cls_row, stream, lens);
  }
  D2S_REQUIRE(hd == kTcHD, D2S_ERR_ARG, "attn_varlen_fwd(bf16): head dim %d unsupported by the tcgen05 kernel (64 only)", hd);
  if (B == 0) return D2S_OK;
  const int Tkp = ceil_div(Tmax, 16) * 16;
  CUtensorMap map_a, map_b;
  int rc = encode_qkv_maps(qkv, B, Tmax, H, Tkp, map_a, map_b);
  if (rc) return rc;
  const int units = B * H;
  if (Tmax <= kTileRows)
    return launch_tc<1, false, 4, true>(map_a, map_b, nullptr, units, Tmax, H, Tkp, scale, 0.0f, out, cls_row, nullptr, qkv, stream, lens);
  return launch_tc<2, false, 8, true>(map_a, map_b, nullptr, units, Tmax, H, Tkp, scale, 0.0f, out, cls_row, nullptr, qkv, stream, lens);
}
