// Validates the fp16 tcgen05 building blocks of ovc_tc.cuh on a B200:
//   D[128 x N] = A[shift .. shift+128) x B^T   (K-major, no swizzle, kind::f16, fp32 accumulate in TMEM)
// (1) single-pass fp16, (2) 3xFP16 split precision with the scaled low-order accumulator: a_hi * [b_hi ; b_lo]^T as ONE
// MMA of width 2N plus a_lo * b_hi^T, (3) row-shifted A
// (a convolution tap), (4) small-magnitude operands (fp16 subnormal range of the high parts).
// nvcc -gencode arch=compute_100a,code=sm_100a -O3 -I openvoice_b200/csrc -o /tmp/tc_f16_test tools/tc_f16_test.cu
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "ovc_conv.cuh"
#include "ovc_tc.cuh"

using namespace ovc;

constexpr int M = 128, N = 64, K = 64, ROWS_A = 160;

// 32 lanes x 8 consecutive fp32 columns: lane i of the warp reads TMEM lane (base_lane + i)
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

__global__ void __launch_bounds__(128) gemm_test(const float* A, const float* B, float* D, int shift, int split) {
  extern __shared__ __align__(128) unsigned char smem[];
  unsigned char* a_hi = smem;                                   // [K/8][ROWS_A][8 halfs]
  unsigned char* a_lo = a_hi + ROWS_A * K * 2;
  unsigned char* b_st = a_lo + ROWS_A * K * 2;                  // [K/8][hi|lo][N][8 halfs]: one 2N-row operand [b_hi ; b_lo]
  uint64_t* bar = reinterpret_cast<uint64_t*>(b_st + 2 * N * K * 2);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
  const int tid = threadIdx.x, warp = tid >> 5;

  for (int e = tid; e < ROWS_A * (K / 8); e += 128) {
    const int row = e / (K / 8), kc = e % (K / 8);
    const float4 v0 = *reinterpret_cast<const float4*>(A + (size_t)row * K + kc * 8);
    const float4 v1 = *reinterpret_cast<const float4*>(A + (size_t)row * K + kc * 8 + 4);
    uint4 hi, lo;
    tc::split_f16x8(v0, v1, 1.f, hi, lo);
    *reinterpret_cast<uint4*>(a_hi + (kc * ROWS_A + row) * 16) = hi;
    *reinterpret_cast<uint4*>(a_lo + (kc * ROWS_A + row) * 16) = lo;
  }
  for (int e = tid; e < N * (K / 8); e += 128) {
    const int row = e / (K / 8), kc = e % (K / 8);
    const float4 v0 = *reinterpret_cast<const float4*>(B + (size_t)row * K + kc * 8);
    const float4 v1 = *reinterpret_cast<const float4*>(B + (size_t)row * K + kc * 8 + 4);
    uint4 hi, lo;
    tc::split_f16x8(v0, v1, 1.f, hi, lo);
    *reinterpret_cast<uint4*>(b_st + ((kc * 2 + 0) * N + row) * 16) = hi;
    *reinterpret_cast<uint4*>(b_st + ((kc * 2 + 1) * N + row) * 16) = lo;
  }
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  if (warp == 0) tc::tmem_alloc(tmem_slot, 128);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc::fence_before();
  __syncthreads();
  tc::fence_after();
  const uint32_t tmem_d = *tmem_slot;

  if (tid == 0) {
    const uint32_t idesc1 = tc::make_idesc_f16(M, N), idesc2 = tc::make_idesc_f16(M, 2 * N);
    const uint32_t lbo_a = ROWS_A * 16, lbo_b = 2 * N * 16, sbo = 128;
    for (int k16 = 0; k16 < K / 16; ++k16) {
      const uint64_t ah = tc::make_desc(tc::smem_addr(a_hi) + (2 * k16) * lbo_a + shift * 16, lbo_a, sbo);
      const uint64_t al = tc::make_desc(tc::smem_addr(a_lo) + (2 * k16) * lbo_a + shift * 16, lbo_a, sbo);
      const uint64_t bs = tc::make_desc(tc::smem_addr(b_st) + (2 * k16) * lbo_b, lbo_b, sbo);
      if (split) {
        tc::mma_f16(tmem_d, ah, bs, idesc2, k16 > 0);       // [main | low] (+)= a_hi * [b_hi ; b_lo]^T
        tc::mma_f16(tmem_d + N, al, bs, idesc1, true);      // low += a_lo * b_hi^T
      } else {
        tc::mma_f16(tmem_d, ah, bs, idesc1, k16 > 0);
      }
    }
    tc::mma_commit(bar);
  }
  mbar_wait(bar, 0);
  tc::fence_after();
  for (int c0 = 0; c0 < N; c0 += 8) {
    float v[8], l[8];
    tmem_ld8(tmem_d + ((uint32_t)(warp * 32) << 16) + c0, v);
    if (split) {
      tmem_ld8(tmem_d + ((uint32_t)(warp * 32) << 16) + N + c0, l);
      for (int i = 0; i < 8; ++i) v[i] = fmaf(l[i], tc::kLoInv, v[i]);
    }
    for (int i = 0; i < 8; ++i) D[(size_t)tid * N + c0 + i] = v[i];
  }
  tc::fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem_d, 128);
}

static double run(int shift, int split, const std::vector<float>& A, const std::vector<float>& B) {
  float *dA, *dB, *dD;
  cudaMalloc(&dA, A.size() * 4); cudaMalloc(&dB, B.size() * 4); cudaMalloc(&dD, M * N * 4);
  cudaMemcpy(dA, A.data(), A.size() * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dB, B.data(), B.size() * 4, cudaMemcpyHostToDevice);
  cudaMemset(dD, 0, M * N * 4);
  const size_t smem = (2 * ROWS_A * K + 2 * N * K) * 2 + 64;
  cudaFuncSetAttribute(gemm_test, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  gemm_test<<<1, 128, smem>>>(dA, dB, dD, shift, split);
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { printf("CUDA error: %s\n", cudaGetErrorString(e)); exit(1); }
  std::vector<float> D(M * N);
  cudaMemcpy(D.data(), dD, M * N * 4, cudaMemcpyDeviceToHost);
  double maxerr = 0, sumsq = 0;
  for (int i = 0; i < M; ++i)
    for (int j = 0; j < N; ++j) {
      double r = 0;
      for (int k = 0; k < K; ++k) r += (double)A[(size_t)(i + shift) * K + k] * (double)B[(size_t)j * K + k];
      maxerr = fmax(maxerr, fabs(r - D[(size_t)i * N + j]));
      sumsq += r * r;
    }
  cudaFree(dA); cudaFree(dB); cudaFree(dD);
  return maxerr / sqrt(sumsq / (M * N));
}

int main() {
  std::vector<float> A(ROWS_A * K), B(N * K);
  srand(1);
  for (auto& v : A) v = (rand() / (float)RAND_MAX) * 2.f - 1.f;
  for (auto& v : B) v = (rand() / (float)RAND_MAX) * 2.f - 1.f;
  printf("fp16 single pass, shift 0 : max err / rms %.3e (expect ~5e-4)\n", run(0, 0, A, B));
  printf("3xFP16 split,     shift 0 : max err / rms %.3e (expect ~1e-6)\n", run(0, 1, A, B));
  printf("3xFP16 split,     shift 3 : max err / rms %.3e\n", run(3, 1, A, B));
  printf("3xFP16 split,     shift 29: max err / rms %.3e\n", run(29, 1, A, B));
  for (auto& v : A) v *= 3e-4f;    // high parts near / below fp16's normal range
  for (auto& v : B) v *= 2e-2f;
  printf("3xFP16 split, small operands (|a| < 3e-4, |b| < 2e-2): max err / rms %.3e\n", run(5, 1, A, B));
  for (auto& v : A) v *= 1e6f;     // |a| up to 300
  printf("3xFP16 split, large operands (|a| < 300): max err / rms %.3e\n", run(5, 1, A, B));
  return 0;
}
