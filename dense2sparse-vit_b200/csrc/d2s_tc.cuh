// tcgen05 / TMEM / TMA / mbarrier PTX wrappers shared by the tensor-core attention kernels (sm_100a).
#pragma once
#include <cuda.h>
#include "d2s_common.cuh"

namespace d2s {

constexpr int kTcHD = 64;        // head dim handled by the tensor-core kernels
constexpr int kTileRows = 128;   // query rows per MMA tile (UMMA M)
constexpr uint32_t kTileBytes = kTileRows * 128;  // 128 rows x 64 bf16

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra LAB_DONE;\n\t"
      "bra LAB_WAIT;\n\t"
      "LAB_DONE:\n\t"
      "}\n" ::"r"(bar), "r"(parity) : "memory");
}
// 1-D bulk copy global -> shared::cta through the TMA unit (no tensor map): `bytes` and both addresses are multiples of 16;
// completion is counted in bytes on `bar`.
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// TMA: 3-D tiled load (coordinates innermost first), completion on an mbarrier
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// 64-bit shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout), SWIZZLE_128B, version 1.
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= 1ull << 46;  // descriptor version (Blackwell)
  d |= 2ull << 61;  // SWIZZLE_128B
  return d;
}
// 32-bit instruction descriptor (cute::UMMA::InstrDescriptor): bf16 x bf16 -> fp32
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int b_mn_major, int a_mn_major = 0) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// Variants with the accumulate flag as an immediate (no setp in the single-thread issue loop: the tcgen05.mma issue
// cadence of one thread is what the short PV product waits on).
template <bool kAccum>
__device__ __forceinline__ void mma_ss_imm(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  if (kAccum)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 1;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc));
  else
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc));
}
template <bool kAccum>
__device__ __forceinline__ void mma_ts_imm(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc) {
  if (kAccum)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 1;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
                 ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc));
  else
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
                 ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc));
}
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void tmem_ld16_nowait(uint32_t addr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(addr));
}
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t addr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(addr));
}
__device__ __forceinline__ void tmem_st16(uint32_t addr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(addr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_ld8_nowait(uint32_t addr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(addr));
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// 2^-d for a non-negative integer-valued d, exactly (exponent-field arithmetic); d >= 127 gives 0
__device__ __forceinline__ float exp2_neg_int(float d) {
  return d < 127.f ? __uint_as_float((uint32_t)(127 - (int)d) << 23) : 0.f;
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st8(uint32_t addr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(addr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));  // first source -> upper half
  return r;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {      // FMNMX3: one issue slot for a three-way maximum
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// byte offset of 16-byte chunk `c` (0..7) of row `r` inside a [rows x 128 B] SWIZZLE_128B tile
__device__ __forceinline__ uint32_t sw128_off(int r, int c) {
  return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4));
}

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}


// ---- packed fp32x2 arithmetic (sm_100: one FFMA2/FMUL2/FADD2 issue slot handles two elements) ----
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t f2_bcast(float c) { return f2_pack(c, c); }

// Exact-erf GELU (nn.GELU(), dynamic_vit.py:162) for two elements:
//     GELU(x) = x Phi(x) = max(x, 0) - a h(a),   a = |x|,   h(a) = Phi(-a) = 0.5 erfcx(a / sqrt 2) exp(-a^2 / 2)
// (for x >= 0: x (1 - h) = x - a h; for x < 0: x h = -a h), so no sign select is needed.  0.5 erfcx(a / sqrt 2) is a degree-8
// polynomial in a on [0, 4 sqrt 2] (relative error 2.2e-4; a is clamped there, where a h < 4e-8), exp(-a^2/2) one MUFU.EX2.
// Error against float64 erf GELU: <= 0.07 bf16 ulp for |x| < 5.6, absolute <= 3.8e-5.  One MUFU and ~10 issue slots per
// element (packed fp32x2 arithmetic) instead of two MUFU and ~23 for the rcp-based erf.
__device__ __forceinline__ uint64_t gelu_erf_pair(uint64_t x) {
  float x0, x1;
  f2_unpack(x, x0, x1);
  const uint64_t a = f2_pack(fminf(fabsf(x0), 5.6568542f), fminf(fabsf(x1), 5.6568542f));
  // r = -0.5 erfcx(a / sqrt 2): the coefficients carry the minus sign of "- a h"
  uint64_t r = f2_fma(f2_bcast(-3.457075050e-06f), a, f2_bcast(9.698495899e-05f));
  r = f2_fma(r, a, f2_bcast(-1.174711513e-03f));
  r = f2_fma(r, a, f2_bcast(8.114228228e-03f));
  r = f2_fma(r, a, f2_bcast(-3.579151344e-02f));
  r = f2_fma(r, a, f2_bcast(1.080985674e-01f));
  r = f2_fma(r, a, f2_bcast(-2.371637582e-01f));
  r = f2_fma(r, a, f2_bcast(3.961593576e-01f));
  r = f2_fma(r, a, f2_bcast(-4.998897713e-01f));
  float e0, e1;
  f2_unpack(f2_mul(f2_mul(x, x), f2_bcast(-0.72134752044448170368f)), e0, e1);   // -x^2/2 * log2(e)
  const uint64_t nh = f2_mul(r, f2_pack(ex2_approx(e0), ex2_approx(e1)));         // -h(a)
  return f2_fma(nh, a, f2_pack(fmaxf(x0, 0.f), fmaxf(x1, 0.f)));
}

// One lane of a fully converged warp (elect.sync).  tcgen05.mma / tcgen05.commit take their operands from UNIFORM registers:
// when the issuing code sits inside `if (lane == 0)` the compiler cannot prove the descriptors warp-uniform and wraps every
// instruction in an ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall loop (~80 cycles per MMA, measured).  Running the issue loop
// warp-uniformly (all 32 lanes: waits, address arithmetic) and predicating only the instruction on elect_one() gives
// straight-line UTCHMMA with uniform-datapath operands.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
// value of lane 0, provably warp-uniform for the compiler
__device__ __forceinline__ int warp_uniform(int v) { return __shfl_sync(0xffffffffu, v, 0); }

// ---- CTA-pair (cluster of 2, tcgen05 cta_group::2) helpers shared by d2s_gemm_pair.cu and d2s_mlp_pair.cu ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local` (a shared::cta address) in the CTA of rank `rank`
__device__ __forceinline__ uint32_t mapa(uint32_t local, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local), "r"(rank));
  return r;
}
// Arrive on a barrier of (possibly) the peer CTA.  Release at CTA scope (the PTX default), as CUTLASS's ClusterBarrier::arrive:
// `.release.cluster` compiles to MEMBAR.ALL.GPU + ERRBAR in front of the arrive (~1000 cycles, measured in the MLP kernel's
// activation stage, twice per chunk).  What these arrives publish is either TMEM reads (ordered by tcgen05.fence +
// tcgen05.wait::ld) or shared-memory writes already fenced with fence.proxy.async (MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load whose completion bytes are counted on a barrier that may live in the peer CTA of the pair
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar_cluster) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster), "r"(c0), "r"(c1) : "memory");
}
template <bool kAccum>
__device__ __forceinline__ void mma2_ss_imm(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  if (kAccum)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 1;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc));
  else
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 1, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                 ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc));
}
// arrive (count 1) on the barrier at the same shared-memory offset in both CTAs of the pair once all prior MMAs retire
__device__ __forceinline__ void mma2_commit_both(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ uint4 ld_nc16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
// 32-byte store (STG.256): a whole sector per thread, for row segments written straight from registers
__device__ __forceinline__ void st_global_v8(void* p, const uint32_t (&r)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]),
               "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ uint32_t add_bf16x2(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("add.rn.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}
// L2-coherent 16-byte load (bypasses L1): data this thread, or another SM, has just written
__device__ __forceinline__ uint4 ld_cg16(const void* p) {
  uint4 r;
  asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
  return r;
}
__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }


typedef CUresult (*GgEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// cuTensorMapEncodeTiled is a DRIVER call: it needs the device's primary context current on the calling thread.  A thread whose
// first CUDA activity is one of these entry points (autograd's backward thread when the node is the only one of the graph)
// has none yet -- the encode then fails with CUDA_ERROR_INVALID_CONTEXT (201).  One runtime call binds it.
static inline void bind_primary_context() {
  static thread_local bool bound = false;
  if (!bound) {
    cudaFree(nullptr);
    bound = true;
  }
}

// d2s_attn_bwd.cu: launches the delta pre-pass of the training attention backwards (stats[..][3] = gout_i . out_i + g_cls . P_0)
int launch_attn_bwd_prep(const void* out, const void* gout, const float* cls_row, const float* g_cls, int B, int T, int H,
                         float* stats, cudaStream_t stream);

static inline GgEncodeFn gg_encode_fn() {
  bind_primary_context();
  static GgEncodeFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<GgEncodeFn>(p);
  }
  return fn;
}


}  // namespace d2s
