// ovc_tc.cuh -- tcgen05 / TMEM helpers (sm_100a inline PTX) for the split-precision tensor-core
// convolution path.  Operand layout used everywhere: K-major, no swizzle ("interleave"):
//   address(row, k) = base + (k / 8) * LBO + (row / 8) * SBO + (row % 8) * 16 + (k % 8) * 2     [f16]
// with SBO = 128 bytes, i.e. rows are uniformly 16 bytes apart inside one 8-channel column
// block, so a convolution tap is just a start-address shift of (tap offset) * 16 bytes.
// One tcgen05.mma.kind::f16 covers K = 16 channels = two column blocks (LBO apart).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ovc {
namespace tc {

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), base_offset [49,52), lbo_mode [52], layout_type [61,64) (0 = no swizzle)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46);
}
// instruction descriptor (cute::UMMA::InstrDescriptor) for kind::f16 with fp16 A and B (a_format = b_format = 0),
// fp32 accumulate (c_format = 1), K-major A and B
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_addr(smem_dst)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // same warp that allocated
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T with fp16 operands (K = 16 per instruction), fp32 accumulation
__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}
// all previously issued MMAs of this thread arrive on the mbarrier when they complete
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_addr(bar)) : "memory");
}
// 16 TMEM lanes x 32 consecutive fp32 columns in the mma-accumulator fragment layout (16x256b.x4): thread i of the
// warp receives, for each 8-column group g = 0..3,
//   r[4g + 0..1] = lane (i / 4),     columns 8g + 2 (i % 4) + {0, 1}
//   r[4g + 2..3] = lane (i / 4) + 8, columns 8g + 2 (i % 4) + {0, 1}
// i.e. four consecutive threads hold 32 contiguous bytes (one DRAM sector) of one output row, so the global loads
// and stores of the epilogue are sector-coalesced without a shared-memory transpose (tools/tmem_ld_probe.cu prints
// this mapping on hardware).  `taddr` carries the first lane (a multiple of 16 inside the warp's 32-lane window).
__device__ __forceinline__ void tmem_ld16x256_x4_issue(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait16(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait16x2(uint32_t (&r)[16], uint32_t (&q)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(q[0]),
                 "+r"(q[1]), "+r"(q[2]), "+r"(q[3]), "+r"(q[4]), "+r"(q[5]), "+r"(q[6]), "+r"(q[7]), "+r"(q[8]), "+r"(q[9]),
                 "+r"(q[10]), "+r"(q[11]), "+r"(q[12]), "+r"(q[13]), "+r"(q[14]), "+r"(q[15])
               :
               : "memory");
}

// true in exactly one lane of a converged warp (elect.sync).  The MMA-issuing warps keep their whole loop converged and
// predicate only the tcgen05.mma / tcgen05.commit on it: operands then stay in uniform registers and ptxas emits one
// predicated UTCHMMA instead of the per-thread ELECT / R2UR / BRA.U.ANY replay loop of a divergent `if (lane == 0)`.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- split precision on fp16 operands ("3xFP16"):  x = hi + lo / 2^11 (+ 2^-23 |x|), hi = fp16(x),
// lo = fp16((x - hi) * 2^11).  The remainder is scaled back into fp16's normal range, so the pair carries 22
// mantissa bits for any |x| < 65504 (absolute floor 2^-36); a*b ~ ah*bh + (al*bh + ah*bl) / 2^11, the two cross
// terms accumulate in their own TMEM accumulator and the epilogue adds them with the 2^-11 factor.  fp16 MMAs run
// at twice the TF32 rate and move half the operand bytes, at the same 11-bit-per-part precision as 3xTF32.
constexpr float kLoScale = 2048.f, kLoInv = 1.f / 2048.f;

// two values -> their hi parts and their lo parts
__device__ __forceinline__ void split_f16x2(float x0, float x1, __half2& hi, __half2& lo) {
  hi = __floats2half2_rn(x0, x1);
  const float2 hf = __half22float2(hi);
  lo = __floats2half2_rn((x0 - hf.x) * kLoScale, (x1 - hf.y) * kLoScale);
}

// 8 consecutive channels of one row (after the input leaky-relu) -> 16 bytes of hi parts + 16 bytes of lo parts
__device__ __forceinline__ void split_f16x8(float4 a, float4 b, float slope, uint4& hi, uint4& lo) {
  float x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float x0 = x[2 * i], x1 = x[2 * i + 1];
    x0 = fmaxf(x0, x0 * slope);   // leaky_relu for 0 <= slope <= 1 (launch_tc checks), bit-identical to the select
    x1 = fmaxf(x1, x1 * slope);
    __half2 hh, ll;
    split_f16x2(x0, x1, hh, ll);
    h[i] = *reinterpret_cast<const uint32_t*>(&hh);
    l[i] = *reinterpret_cast<const uint32_t*>(&ll);
  }
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}

}  // namespace tc
}  // namespace ovc
