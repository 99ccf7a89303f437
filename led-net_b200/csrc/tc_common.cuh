// PTX wrappers shared by the tcgen05 kernels (conv_tc.cu, stem_tc.cu): mbarrier, TMA, tcgen05 MMA /
// TMEM load, UMMA shared-memory descriptors, and the 128 B XOR swizzle used for epilogue staging.
#pragma once
#include <cuda.h>

#include "kernels.h"

namespace ledb {
// cuTensorMapEncodeTiled through the runtime's driver entry point (conv_tc.cu): element type = 2-byte units, swizzle
// 128 / 64 / 32 B for a box of 64 / 32 / 16 units
int tc_encode_tiled(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box, int kc);
// weight gradient on the tensor cores (wgrad_tc.cu)
bool wgrad_tc_eligible(int N, int H, int W, int Cin, int Cout, int k, int stride, int passes);
int64_t wgrad_tc_workspace_bytes(int N, int H, int W, int Cin, int Cout, int k, int stride, int passes);
int launch_wgrad_tc(const float* x, const float* dy, float* dw, int N, int H, int W, int Cin, int Cout, int k, int stride,
                    int passes, void* workspace, cudaStream_t st);
namespace tc {

__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_tensormap(const void* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (visible as a launch failure) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 28)) __trap();
  }
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
               ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
               ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
// generic-proxy shared-memory writes (st.shared) -> visible to the async proxy (UMMA operand reads)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// Predicated forms: the whole warp executes the (warp-uniform) address arithmetic, only the lane
// whose `pred` is non-zero issues - no divergent region around the MMA loop, so descriptors can stay
// in uniform registers.
__device__ __forceinline__ void tc_commit_if(uint64_t* bar, uint32_t pred) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
      ::"r"(smem_u32(bar)), "r"(pred) : "memory");
}
__device__ __forceinline__ void tc_mma_if(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate, uint32_t pred) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(pred) : "memory");
}
// Same, with the two 64-bit shared-memory descriptors passed as (low, high) words: the high words are
// loop constants and the low words advance by immediates, so the issue loop needs no 64-bit arithmetic.
__device__ __forceinline__ void tc_mma_if2(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                           uint32_t idesc, uint32_t accumulate, uint32_t pred) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "setp.ne.b32 q, %7, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate), "r"(pred) : "memory");
}
// Unpredicated form for a region entered by ONE elected lane (`if (elect_one())`): ptxas then knows a single
// thread is active and emits the MMA without the ELECT / BRA.U.ANY waterfall loop a per-lane predicate costs.
__device__ __forceinline__ void tc_mma2(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate) : "memory");
}
// same, accumulate always on (no predicate operand to materialise)
__device__ __forceinline__ void tc_mma2_acc(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                            uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.eq.b32 p, 0, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc) : "memory");
}
// ---- kind::tf32 (training path, conv_tc.cu TF32 instantiations and wgrad_tc.cu): A/B are fp32 words in shared memory of which
// the tensor core uses sign + 8-bit exponent + 10-bit mantissa; K = 8 per instruction (32 B of a K-major row, the same byte
// geometry as K = 16 of bf16), fp32 accumulation in TMEM.
__device__ __forceinline__ void tc_mma2_tf32(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_mma2_acc_tf32(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                                 uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.eq.b32 p, 0, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc) : "memory");
}
// instruction descriptor, kind::tf32: D fp32, A/B tf32 (format 2), M = 128, N = n; a_mn / b_mn = 1 selects an MN-major operand
// (bits 15 / 16: the weight-gradient GEMM reads both operands with the reduction dimension - pixels - as shared-memory rows)
__device__ __forceinline__ uint32_t make_idesc_tf32_m128(int n, uint32_t a_mn = 0, uint32_t b_mn = 0) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (a_mn << 15) | (b_mn << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(128 >> 4) << 24);
}
// round-to-nearest fp32 -> tf32 (result is an fp32 bit pattern with the low 13 mantissa bits cleared)
__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t cols) {  // the same warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
}

// UMMA instruction descriptor, kind::f16: D fp32, A/B bf16, both K-major, M = 128, N = n
// (cute/arch/mma_sm100_desc.hpp InstrDescriptor: c_format [4,6), a_format [7,10), b_format [10,13),
// n_dim>>3 [17,23), m_dim>>4 [24,29)).
__device__ __forceinline__ uint32_t make_idesc_bf16_m128(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
// UMMA shared-memory descriptor, K-major operand, swizzled rows (cute SmemDescriptor): start>>4 [0,14),
// LBO>>4 [16,30), SBO>>4 [32,46), version=1 [46,48), base_offset [49,52), layout type [61,64)
// (2 = 128 B swizzle, 4 = 64 B, 6 = 32 B).  The high word is constant per operand; MMA loops only
// rebuild the low word (start address).
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo_bytes, uint32_t layout_type) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | ((layout_type & 7u) << 29);
}
__device__ __forceinline__ uint64_t make_desc(uint32_t hi, uint32_t saddr) {
  const uint32_t lo = ((saddr >> 4) & 0x3FFFu) | (1u << 16);   // LBO (unused for swizzled K-major) = 1
  return ((uint64_t)hi << 32) | lo;
}

// 128 B XOR swizzle of a linear byte offset (bank-conflict-free epilogue staging; base 1024 B aligned)
__device__ __forceinline__ uint32_t swz(uint32_t a) { return a ^ (((a >> 7) & 7u) << 4); }

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_f16x2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_f16x2_sat(float a, float b) {   // a -> low half, b -> high half
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) { float2 t = __bfloat1622float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
}

}  // namespace tc
}  // namespace ledb
