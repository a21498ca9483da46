// How accurate is the fp32 accumulation of tcgen05.mma.kind::tf32 over MANY accumulation steps?
// D[128 x 64] = A[128 x K] * B[64 x K]^T with 3xTF32, K = 2048 (256 MMA steps per pass), operands staged
// chunk by chunk (K=32 per stage).  Variants: (0) one accumulator for all three passes,
// (1) the two low-order passes in their own accumulator, (2) as 1 plus main accumulator alternating
// between two TMEM regions.  Reports max|err|/rms(ref) and rms(err)/rms(ref) against fp64.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "ovc_conv.cuh"
#include "ovc_tc.cuh"
using namespace ovc;
constexpr int M = 128, N = 64, KC = 32;

// the kind::tf32 building blocks this probe needs (the library's kernels use kind::f16 only)
// instruction descriptor (cute::UMMA::InstrDescriptor) for kind::tf32, fp32 accumulate, K-major A and B
__host__ __device__ constexpr uint32_t make_idesc_tf32(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]^T, issued by ONE thread
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
      : "memory");
}
// split an fp32 into a tf32-exact high part and the fp32 remainder (3xTF32: a*b ~ ah*bh + al*bh + ah*bl)
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  hi = __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
  lo = x - hi;
}
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

__global__ void __launch_bounds__(128) k(const float* A, const float* B, float* D, int K, int variant) {
  extern __shared__ __align__(128) unsigned char smem[];
  float* a_hi = reinterpret_cast<float*>(smem);
  float* a_lo = a_hi + M * KC;
  float* b_hi = a_lo + M * KC;
  float* b_lo = b_hi + N * KC;
  uint64_t* bar = reinterpret_cast<uint64_t*>(b_lo + N * KC);
  uint32_t* slot = reinterpret_cast<uint32_t*>(bar + 1);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) { mbar_init(bar, 1); fence_mbar_init(); }
  if (warp == 0) tc::tmem_alloc(slot, 256);
  tc::fence_before(); __syncthreads(); tc::fence_after();
  const uint32_t tm = *slot;
  const uint32_t idesc = make_idesc_tf32(M, N);
  int phase = 0;
  for (int k0 = 0; k0 < K; k0 += KC) {
    for (int e = tid; e < M * KC; e += 128) {
      const int row = e / KC, kk = e % KC; float hi, lo; split_tf32(A[(size_t)row * K + k0 + kk], hi, lo);
      a_hi[((kk / 4) * M + row) * 4 + (kk % 4)] = hi; a_lo[((kk / 4) * M + row) * 4 + (kk % 4)] = lo;
    }
    for (int e = tid; e < N * KC; e += 128) {
      const int row = e / KC, kk = e % KC; float hi, lo; split_tf32(B[(size_t)row * K + k0 + kk], hi, lo);
      b_hi[((kk / 4) * N + row) * 4 + (kk % 4)] = hi; b_lo[((kk / 4) * N + row) * 4 + (kk % 4)] = lo;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc::fence_before(); __syncthreads(); tc::fence_after();
    if (tid == 0) {
      for (int k8 = 0; k8 < KC / 8; ++k8) {
        const int step = k0 / 8 + k8;
        const uint64_t ah = tc::make_desc(tc::smem_addr(a_hi) + 2 * k8 * M * 16, M * 16, 128);
        const uint64_t al = tc::make_desc(tc::smem_addr(a_lo) + 2 * k8 * M * 16, M * 16, 128);
        const uint64_t bh = tc::make_desc(tc::smem_addr(b_hi) + 2 * k8 * N * 16, N * 16, 128);
        const uint64_t bl = tc::make_desc(tc::smem_addr(b_lo) + 2 * k8 * N * 16, N * 16, 128);
        const uint32_t d_main = tm + ((variant == 2) ? (step & 1) * 64 : 0);
        const uint32_t d_lo = (variant >= 1) ? tm + 128 : d_main;
        mma_tf32(d_main, ah, bh, idesc, variant == 2 ? step >= 2 : step >= 1);
        mma_tf32(d_lo, al, bh, idesc, variant >= 1 ? step >= 1 : true);
        mma_tf32(d_lo, ah, bl, idesc, true);
      }
      tc::mma_commit(bar);
    }
    mbar_wait(bar, phase); phase ^= 1;
    tc::fence_after();
  }
  for (int c0 = 0; c0 < N; c0 += 8) {
    float v[8], w[8], u[8];
    tmem_ld8(tm + ((uint32_t)(warp * 32) << 16) + c0, v);
    if (variant == 2) { tmem_ld8(tm + ((uint32_t)(warp * 32) << 16) + 64 + c0, u); for (int i = 0; i < 8; ++i) v[i] += u[i]; }
    if (variant >= 1) { tmem_ld8(tm + ((uint32_t)(warp * 32) << 16) + 128 + c0, w); for (int i = 0; i < 8; ++i) v[i] += w[i]; }
    for (int i = 0; i < 8; ++i) D[(size_t)tid * N + c0 + i] = v[i];
  }
  tc::fence_before(); __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tm, 256);
}

int main() {
  const int K = 2048;
  std::vector<float> A((size_t)M * K), B((size_t)N * K);
  srand(3);
  for (auto& v : A) v = (rand() / (float)RAND_MAX) * 2.f - 1.f;
  for (auto& v : B) v = (rand() / (float)RAND_MAX) * 2.f - 1.f;
  float *dA, *dB, *dD;
  cudaMalloc(&dA, A.size() * 4); cudaMalloc(&dB, B.size() * 4); cudaMalloc(&dD, M * N * 4);
  cudaMemcpy(dA, A.data(), A.size() * 4, cudaMemcpyHostToDevice);
  cudaMemcpy(dB, B.data(), B.size() * 4, cudaMemcpyHostToDevice);
  std::vector<double> ref((size_t)M * N);
  double rms = 0;
  for (int i = 0; i < M; ++i) for (int j = 0; j < N; ++j) {
    double r = 0; for (int kk = 0; kk < K; ++kk) r += (double)A[(size_t)i * K + kk] * B[(size_t)j * K + kk];
    ref[(size_t)i * N + j] = r; rms += r * r;
  }
  rms = sqrt(rms / (M * N));
  // fp32 sequential accumulation on the host for comparison
  double e32 = 0;
  for (int i = 0; i < M; ++i) for (int j = 0; j < N; ++j) {
    float r = 0; for (int kk = 0; kk < K; ++kk) r = fmaf(A[(size_t)i * K + kk], B[(size_t)j * K + kk], r);
    e32 = fmax(e32, fabs(r - ref[(size_t)i * N + j]));
  }
  printf("host fp32 fmaf chain: max err / rms = %.3e\n", e32 / rms);
  const size_t smem = (2 * M * KC + 2 * N * KC) * 4 + 64;
  cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  for (int variant = 0; variant < 3; ++variant) {
    k<<<1, 128, smem>>>(dA, dB, dD, K, variant);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { printf("CUDA error %s\n", cudaGetErrorString(e)); return 1; }
    std::vector<float> D((size_t)M * N);
    cudaMemcpy(D.data(), dD, D.size() * 4, cudaMemcpyDeviceToHost);
    double mx = 0, se = 0, bias = 0;
    for (size_t i = 0; i < D.size(); ++i) { const double d = D[i] - ref[i]; mx = fmax(mx, fabs(d)); se += d * d; bias += d * (ref[i] > 0 ? 1 : -1); }
    printf("variant %d: max err / rms = %.3e, rms err / rms = %.3e, mean signed err toward |ref| = %.3e\n", variant, mx / rms,
           sqrt(se / D.size()) / rms, bias / D.size() / rms);
  }
  return 0;
}
