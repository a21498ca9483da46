// ovc_conv.cuh -- the one convolution kernel family of the tone-colour-converter hot path.
//
// Every conv on ToneColorConverter.convert -> SynthesizerTrn.voice_conversion (198 Conv1d +
// 4 ConvTranspose1d; SURVEY.md section 0.2) is an instance of conv1d_f32<> below: an fp32
// implicit GEMM  Y[row, t] = sum_{ci,k} W[row, ci, k] * act(X[ci, t + (k-(K-1)/2)*DIL])
// with the surrounding elementwise work of the reference fused into the prologue
// (leaky_relu while staging X) and the epilogue (bias, speaker conditioning + tanh*sigmoid
// gate, residual/skip accumulation, reparameterisation noise, coupling update, MRF averaging,
// polyphase scatter of the transposed convs).
//
// Mapping to B200 (sm_100a):
//  * CTA tile = (32*WM) output rows x (64*WN) time steps, one warp per 32x64 sub-tile, lanes as
//    4 (rows) x 8 (time), 8x(4+4) accumulators per thread -> FFMA-bound inner loop (the path is
//    a dense fp32 contraction: SURVEY.md section 8d).
//  * Weights are pre-packed [row_tile][ci][k][rows] so one ci-chunk of a row tile is ONE
//    contiguous blob, fetched by a single TMA bulk copy (cp.async.bulk -> UBLKCP) that signals
//    an mbarrier; two stages.
//  * Activations are staged by 16-byte cp.async with zero-fill: out-of-range time steps and
//    steps past the utterance length arrive as zeros, which IS the reference's zero padding and
//    its x_mask multiplications.  leaky_relu is applied once per staged element in smem.
//  * The inner loop keeps a sliding window of the X row in registers (aligned LDS.128, reused by
//    all K taps; dilated taps simply index further into the same window) and broadcasts weight
//    fragments with LDS.128 -- ~8 shared loads per 100 FFMA.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ovc {

enum EpiKind : int {
  EPI_LINEAR = 0,   // y = (conv + bias [+ res] [+ y_old]) * scale         (pre, conv_pre, ResBlock1 convs)
  EPI_GATE = 1,     // y = tanh(a + g_a) * sigmoid(b + g_b)               (WN in_layer; commons.py:100-107)
  EPI_RESSKIP = 2,  // x += rs[:H] ; skip (+)= rs[H:]                     (WN res_skip; modules.py:203-209)
  EPI_PROJ = 3,     // z = m + noise * tau * exp(logs)                    (enc_q.proj; models.py:218-220)
  EPI_COUPLE = 4,   // x1 = x1 +/- m                                      (coupling post; modules.py:441-454)
  EPI_UPS8 = 5,     // polyphase ConvTranspose1d stride 8 (k=16, p=4)     (models.py:245-256, :279)
  EPI_UPS2 = 6      // polyphase ConvTranspose1d stride 2 (k=4,  p=1)
};

enum : int { F_ACCUM = 1, F_FIRST = 2 };

// per-call scalars that live in device memory so that a captured launch sequence (CUDA graph) can be replayed with new values
struct CallParams { unsigned long long seed; float tau; float pad; };

struct ConvArgs {
  // input activations, [B][cin][x_pitch] (time fastest)
  const float* x; long long x_bs; int x_pitch; int cin;
  // packed weights [row_tiles][n_chunks*CI_CH][K][CO_T]; bias per packed row (+ b*bias_bs)
  const float* w; const float* bias; long long bias_bs;
  int n_chunks;
  // primary output / in-place target
  float* y; long long y_bs; int y_pitch;
  // secondary tensors (residual for LINEAR, skip accumulator for RESSKIP, noise for PROJ)
  const float* r; long long r_bs; int r_pitch;
  float* s; long long s_bs; int s_pitch;
  // per-utterance valid lengths (frames); NULL -> tmax.  limits = base * mul
  const long long* lens_in; const long long* lens_out; int tmax; int mul_in; int mul_out;
  float slope;      // leaky_relu slope applied to X while staging (1 = identity)
  float scale;      // LINEAR: multiply the result (1/3 for the last MRF accumulation, else 1)
  float tau;        // PROJ
  float sign;       // COUPLE: +1 forward, -1 reverse
  int flags;        // F_ACCUM, F_FIRST
  int split;        // RESSKIP: rows < split update x, rows >= split go to skip[row-split]
  unsigned long long seed;   // PROJ without explicit noise
  const CallParams* callp;   // PROJ: when set, seed and tau are read from here instead (graph replay)
};

// ---------------------------------------------------------------------------------------------
// PTX helpers (sm_100a)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// A wait that cannot complete is a protocol bug: trap after ~2 s instead of hanging the device (the launch then fails
// with an error the host reports), cost: one clock read per FAILED poll.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) __trap();
  }
}
// TMA 1-D bulk copy global -> shared, completion counted in bytes on an mbarrier.
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void cp_async16_zfill(void* dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(src_bytes)
               : "memory");
}
__device__ __forceinline__ void cp_async4_zfill(void* dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(src_bytes)
               : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

__device__ __forceinline__ float lrelu(float v, float slope) { return v > 0.f ? v : v * slope; }
__device__ __forceinline__ float sigmoidf_acc(float v) { return 1.f / (1.f + expf(-v)); }

// Philox4x32-10 -> one standard normal per (b, channel, t) counter (used when no explicit noise
// tensor is supplied; the reference draws torch.randn_like at models.py:220).
__device__ __forceinline__ float philox_normal(unsigned long long seed, uint32_t c0, uint32_t c1, uint32_t c2) {
  uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
  uint32_t x0 = c0, x1 = c1, x2 = c2, x3 = 0x0B200u;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, x0), lo0 = 0xD2511F53u * x0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, x2), lo1 = 0xCD9E8D57u * x2;
    const uint32_t y0 = hi1 ^ x1 ^ k0, y1 = lo1, y2 = hi0 ^ x3 ^ k1, y3 = lo0;
    x0 = y0; x1 = y1; x2 = y2; x3 = y3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  const float u1 = (static_cast<float>(x0 >> 8) + 0.5f) * (1.0f / 16777216.0f);
  const float u2 = (static_cast<float>(x1 >> 8) + 0.5f) * (1.0f / 16777216.0f);
  return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}

// ---------------------------------------------------------------------------------------------
// compile-time tap geometry
// ---------------------------------------------------------------------------------------------
__host__ __device__ constexpr int floor4(int v) { return v >= 0 ? (v / 4) * 4 : -(((-v) + 3) / 4) * 4; }

template <int K, int DIL, int NG>
struct TapGeom {
  static constexpr int HALF = (K - 1) / 2;
  static constexpr int TPG = (K + NG - 1) / NG;  // taps per group
  __host__ __device__ static constexpr int off(int k) { return (k - HALF) * DIL; }
  __host__ __device__ static constexpr int k_lo(int g) { return g * TPG; }
  __host__ __device__ static constexpr int k_hi(int g) { return (g + 1) * TPG < K ? (g + 1) * TPG : K; }  // excl
  __host__ __device__ static constexpr int lo(int g) { return floor4(off(k_lo(g))); }
  __host__ __device__ static constexpr int nvec(int g) { return (off(k_hi(g) - 1) + 3 - lo(g)) / 4 + 1; }
  static constexpr int HL = -lo(0);                                   // left halo (multiple of 4)
  static constexpr int HR = lo(NG - 1) + 4 * nvec(NG - 1) - 4;        // right halo (multiple of 4)
};

template <int K_, int DIL_, int WM_, int WN_, int CI_CH_, int EPI_, int NG_ = 1, int XALIGN_ = 16>
struct ConvCfg {
  static constexpr int K = K_, DIL = DIL_, WM = WM_, WN = WN_, CI_CH = CI_CH_, EPI = EPI_, NG = NG_;
  static constexpr int XALIGN = XALIGN_;
  using G = TapGeom<K, DIL, NG>;
  static constexpr int CO_T = 32 * WM;
  static constexpr int T_T = 64 * WN;
  static constexpr int THREADS = 32 * WM * WN;
  static constexpr int HL = G::HL, HR = G::HR;
  static constexpr int XW = HL + T_T + HR;               // smem row width in floats (multiple of 4)
  static constexpr int W_STAGE = CI_CH * K * CO_T;       // floats
  static constexpr int X_STAGE = CI_CH * XW;             // floats (compact)
  static constexpr size_t SMEM_BYTES = 16 + sizeof(float) * 2 * (W_STAGE + X_STAGE);
  static constexpr int MIN_BLOCKS = (THREADS >= 256) ? 2 : (THREADS >= 128 ? 3 : 4);
};

typedef unsigned long long u64;
// d.lo += a.lo * x ; d.hi += a.hi * x  -- ptxas folds the {x, x} pack into the FFMA2 scalar-broadcast
// operand form (SASS: FFMA2 Rd, Ra.F32x2.HI_LO, Rx.F32, Rd.F32x2.HI_LO), so it costs no instruction.
__device__ __forceinline__ void fma2_bcast(u64& d, const u64 a, const float x) {
  u64 xx;
  asm("mov.b64 %0, {%1, %1};" : "=l"(xx) : "f"(x));
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(a), "l"(xx));
}

// Polyphase structure of the transposed convs (row r of a thread's 8 packed rows, pair rp = rows 2rp, 2rp+1):
//   stride 8: r = phase p; taps used: p<4 -> {x[n-1], x[n]}, p>=4 -> {x[n], x[n+1]}
//   stride 2: r = 2*i + p; p=0 -> {x[n-1], x[n]}, p=1 -> {x[n], x[n+1]}
// true where tap k is zero for both rows of pair rp, so the packed FMA can be skipped
template <int EPI>
__host__ __device__ constexpr bool pair_is_zero(int k, int rp) {
  if (EPI == EPI_UPS8) return (k == 0 && rp >= 2) || (k == 2 && rp < 2);
  return false;   // stride-2 polyphase rows alternate inside a pair: the packed zeros are multiplied
}

// one tap group of one 4-wide time chunk, packed: acc[rp][j] holds rows (2rp, 2rp+1) at time j
template <class C, int G>
__device__ __forceinline__ void tap_group(u64 (&acc)[4][4], const float* __restrict__ xrow,
                                          const float* __restrict__ wrow) {
  using TG = typename C::G;
  constexpr int NV = TG::nvec(G);
  constexpr int LO = TG::lo(G);
  float win[4 * NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float4 v = *reinterpret_cast<const float4*>(xrow + LO + 4 * i);
    win[4 * i + 0] = v.x; win[4 * i + 1] = v.y; win[4 * i + 2] = v.z; win[4 * i + 3] = v.w;
  }
#pragma unroll
  for (int k = TG::k_lo(G); k < TG::k_hi(G); ++k) {
    const ulonglong2 wa = *reinterpret_cast<const ulonglong2*>(wrow + k * C::CO_T);
    const ulonglong2 wb = *reinterpret_cast<const ulonglong2*>(wrow + k * C::CO_T + 4);
    const u64 w2[4] = {wa.x, wa.y, wb.x, wb.y};   // rows (0,1) (2,3) (4,5) (6,7)
    const int base = TG::off(k) - LO;
#pragma unroll
    for (int rp = 0; rp < 4; ++rp) {
      if (pair_is_zero<C::EPI>(k, rp)) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) fma2_bcast(acc[rp][j], w2[rp], win[base + j]);
    }
  }
}

template <class C>
__device__ __forceinline__ void compute_chunk(u64 (&acc)[2][4][4], const float* __restrict__ xs,
                                              const float* __restrict__ ws, int tb, int cb) {
#pragma unroll 1
  for (int ci = 0; ci < C::CI_CH; ++ci) {
    const float* wrow = ws + ci * (C::K * C::CO_T) + cb;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const float* xrow = xs + ci * C::XW + C::HL + tb + 32 * c;
      tap_group<C, 0>(acc[c], xrow, wrow);
      if constexpr (C::NG >= 2) tap_group<C, 1>(acc[c], xrow, wrow);
      if constexpr (C::NG >= 3) tap_group<C, 2>(acc[c], xrow, wrow);
      if constexpr (C::NG >= 4) tap_group<C, 3>(acc[c], xrow, wrow);
    }
  }
}

// stage one ci-chunk of X: rows [ci0, ci0+CI_CH), time [t0-HL, t0+T_T+HR)
template <class C>
__device__ __forceinline__ void stage_x_async(float* xs, const float* __restrict__ xb, int x_pitch, int cin,
                                              int ci0, int t0, int lim) {
  if constexpr (C::XALIGN == 16) {
    constexpr int VPR = C::XW / 4;
    constexpr int NVEC = C::CI_CH * VPR;
    for (int v = threadIdx.x; v < NVEC; v += C::THREADS) {
      const int row = v / VPR, col = v - row * VPR;
      const int t = t0 - C::HL + 4 * col;
      const int ci = ci0 + row;
      int nb = 0;
      if (ci < cin && t >= 0 && t < lim) nb = (lim - t >= 4) ? 16 : 4 * (lim - t);
      const float* src = nb ? xb + (size_t)ci * x_pitch + t : xb;
      cp_async16_zfill(xs + row * C::XW + 4 * col, src, nb);
    }
  } else {
    constexpr int NEL = C::CI_CH * C::XW;
    for (int e = threadIdx.x; e < NEL; e += C::THREADS) {
      const int row = e / C::XW, col = e - row * C::XW;
      const int t = t0 - C::HL + col;
      const int ci = ci0 + row;
      const bool ok = (ci < cin && t >= 0 && t < lim);
      const float* src = ok ? xb + (size_t)ci * x_pitch + t : xb;
      cp_async4_zfill(xs + row * C::XW + col, src, ok ? 4 : 0);
    }
  }
}
// leaky_relu on exactly the elements this thread staged (visible to it after cp.async.wait_all)
template <class C>
__device__ __forceinline__ void stage_x_activate(float* xs, float slope) {
  if (slope == 1.f) return;
  if constexpr (C::XALIGN == 16) {
    constexpr int NVEC = C::CI_CH * (C::XW / 4);
    float4* p = reinterpret_cast<float4*>(xs);
    for (int v = threadIdx.x; v < NVEC; v += C::THREADS) {
      float4 q = p[v];
      q.x = lrelu(q.x, slope); q.y = lrelu(q.y, slope); q.z = lrelu(q.z, slope); q.w = lrelu(q.w, slope);
      p[v] = q;
    }
  } else {
    constexpr int NEL = C::CI_CH * C::XW;
    for (int e = threadIdx.x; e < NEL; e += C::THREADS) xs[e] = lrelu(xs[e], slope);
  }
}

// ---------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------
template <class C>
__global__ void __launch_bounds__(C::THREADS, C::MIN_BLOCKS) conv1d_f32(const ConvArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
  float* wsm = reinterpret_cast<float*>(smem_raw + 16);
  float* xsm = wsm + 2 * C::W_STAGE;

  const int b = blockIdx.z;
  const int t0 = blockIdx.x * C::T_T;
  const int base_in = a.lens_in ? (int)min((long long)a.tmax, a.lens_in[b]) : a.tmax;
  const int base_out = a.lens_out ? (int)min((long long)a.tmax, a.lens_out[b]) : a.tmax;
  const int in_lim = base_in * a.mul_in;
  const int out_lim = base_out * a.mul_out;   // in units of this kernel's time axis
  if (t0 >= out_lim) return;                  // whole tile is padding (block-uniform)

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int warp_m = warp % C::WM, warp_n = warp / C::WM;
  const int lane_co = lane >> 3, lane_t = lane & 7;
  const int cb = warp_m * 32 + lane_co * 8;   // first of this thread's 8 packed rows in the tile
  const int tb = warp_n * 64 + lane_t * 4;    // first of this thread's time chunk 0 (chunk 1 = +32)

  const float* xb = a.x + (size_t)b * a.x_bs;
  const float* wtile = a.w + (size_t)blockIdx.y * a.n_chunks * C::W_STAGE;
  constexpr uint32_t W_BYTES = C::W_STAGE * sizeof(float);

  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    fence_mbar_init();
  }
  __syncthreads();

  // prologue: chunk 0
  if (tid == 0) {
    mbar_expect_tx(&bars[0], W_BYTES);
    tma_bulk_g2s(wsm, wtile, W_BYTES, &bars[0]);
  }
  stage_x_async<C>(xsm, xb, a.x_pitch, a.cin, 0, t0, in_lim);
  cp_async_wait_all();
  stage_x_activate<C>(xsm, a.slope);
  __syncthreads();

  u64 accw[2][4][4];
#pragma unroll
  for (int c = 0; c < 2; ++c)
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int j = 0; j < 4; ++j) accw[c][r][j] = 0ull;

  const int n_chunks = a.n_chunks;
  for (int ch = 0; ch < n_chunks; ++ch) {
    const int s = ch & 1;
    if (ch + 1 < n_chunks) {   // prefetch next chunk into the other stage (freed by the barrier below)
      if (tid == 0) {
        mbar_expect_tx(&bars[s ^ 1], W_BYTES);
        tma_bulk_g2s(wsm + (s ^ 1) * C::W_STAGE, wtile + (size_t)(ch + 1) * C::W_STAGE, W_BYTES, &bars[s ^ 1]);
      }
      stage_x_async<C>(xsm + (s ^ 1) * C::X_STAGE, xb, a.x_pitch, a.cin, (ch + 1) * C::CI_CH, t0, in_lim);
    }
    mbar_wait(&bars[s], (ch >> 1) & 1);
    compute_chunk<C>(accw, xsm + s * C::X_STAGE, wsm + s * C::W_STAGE, tb, cb);
    if (ch + 1 < n_chunks) {
      cp_async_wait_all();
      stage_x_activate<C>(xsm + (s ^ 1) * C::X_STAGE, a.slope);
    }
    __syncthreads();
  }

  float acc[2][8][4];
#pragma unroll
  for (int c = 0; c < 2; ++c)
#pragma unroll
    for (int rp = 0; rp < 4; ++rp)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        acc[c][2 * rp][j] = __uint_as_float((unsigned)(accw[c][rp][j] & 0xffffffffull));
        acc[c][2 * rp + 1][j] = __uint_as_float((unsigned)(accw[c][rp][j] >> 32));
      }

  // ------------------------------------------------------------------ epilogue
  const int row0 = blockIdx.y * C::CO_T + cb;   // first packed row of this thread
  if constexpr (C::EPI == EPI_LINEAR) {
    const float* bias = a.bias + (size_t)b * a.bias_bs + row0;
    float* yb = a.y + (size_t)b * a.y_bs;
    const float* rb = a.r ? a.r + (size_t)b * a.r_bs : nullptr;
    const bool accum = a.flags & F_ACCUM;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int t = t0 + tb + 32 * c;
      if (t >= out_lim) continue;
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const float bv = bias[r];
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = acc[c][r][j] + bv;
        float* yp = yb + (size_t)(row0 + r) * a.y_pitch + t;
        if (t + 3 < out_lim) {
          if (rb) {
            const float4 q = *reinterpret_cast<const float4*>(rb + (size_t)(row0 + r) * a.r_pitch + t);
            v[0] += q.x; v[1] += q.y; v[2] += q.z; v[3] += q.w;
          }
          if (accum) {
            const float4 q = *reinterpret_cast<const float4*>(yp);
            v[0] = q.x + v[0]; v[1] = q.y + v[1]; v[2] = q.z + v[2]; v[3] = q.w + v[3];
          }
          if (a.scale != 1.f) {
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = v[j] * a.scale;
          }
          *reinterpret_cast<float4*>(yp) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (t + j < out_lim) {
              float u = v[j];
              if (rb) u += rb[(size_t)(row0 + r) * a.r_pitch + t + j];
              if (accum) u = yp[j] + u;
              if (a.scale != 1.f) u = u * a.scale;
              yp[j] = u;
            }
          }
        }
      }
    }
  } else if constexpr (C::EPI == EPI_GATE) {
    // packed rows: r<4 -> tanh half of channel (row0/2 + r), r>=4 -> its sigmoid partner
    const float* gb = a.bias + (size_t)b * a.bias_bs + row0;
    const int ch0 = row0 / 2;
    float* yb = a.y + (size_t)b * a.y_bs;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int t = t0 + tb + 32 * c;
      if (t >= out_lim) continue;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
          v[j] = tanhf(acc[c][r][j] + gb[r]) * sigmoidf_acc(acc[c][r + 4][j] + gb[r + 4]);
        float* yp = yb + (size_t)(ch0 + r) * a.y_pitch + t;
        if (t + 3 < out_lim) {
          *reinterpret_cast<float4*>(yp) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (t + j < out_lim) yp[j] = v[j];
        }
      }
    }
  } else if constexpr (C::EPI == EPI_RESSKIP) {
    const float* bias = a.bias + row0;
    const bool to_x = (row0 < a.split);   // tile-uniform (split is a multiple of CO_T or 0)
    float* base = to_x ? a.y + (size_t)b * a.y_bs + (size_t)row0 * a.y_pitch
                       : a.s + (size_t)b * a.s_bs + (size_t)(row0 - a.split) * a.s_pitch;
    const int pitch = to_x ? a.y_pitch : a.s_pitch;
    const bool add = to_x || !(a.flags & F_FIRST);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int t = t0 + tb + 32 * c;
      if (t >= out_lim) continue;
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        float* yp = base + (size_t)r * pitch + t;
        const float bv = bias[r];
        if (t + 3 < out_lim) {
          float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
          if (add) q = *reinterpret_cast<const float4*>(yp);
          q.x += acc[c][r][0] + bv; q.y += acc[c][r][1] + bv; q.z += acc[c][r][2] + bv; q.w += acc[c][r][3] + bv;
          *reinterpret_cast<float4*>(yp) = q;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (t + j < out_lim) yp[j] = (add ? yp[j] : 0.f) + (acc[c][r][j] + bv);
        }
      }
    }
  } else if constexpr (C::EPI == EPI_PROJ) {
    // packed rows: r<4 -> m of channel (row0/2 + r), r>=4 -> logs of the same channel
    const float* bias = a.bias + row0;
    const int ch0 = row0 / 2;
    float* yb = a.y + (size_t)b * a.y_bs;
    const float* nb = a.r ? a.r + (size_t)b * a.r_bs : nullptr;
    const unsigned long long seed = a.callp ? a.callp->seed : a.seed;
    const float tau = a.callp ? a.callp->tau : a.tau;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int t = t0 + tb + 32 * c;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (t + j < out_lim) {
            const float m = acc[c][r][j] + bias[r];
            const float logs = acc[c][r + 4][j] + bias[r + 4];
            const float nz = nb ? nb[(size_t)(ch0 + r) * a.r_pitch + t + j]
                                : philox_normal(seed, (uint32_t)b, (uint32_t)(ch0 + r), (uint32_t)(t + j));
            yb[(size_t)(ch0 + r) * a.y_pitch + t + j] = m + nz * tau * expf(logs);
          }
        }
      }
    }
  } else if constexpr (C::EPI == EPI_COUPLE) {
    const float* bias = a.bias + row0;
    float* yb = a.y + (size_t)b * a.y_bs;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int t = t0 + tb + 32 * c;
      if (t >= out_lim) continue;
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        float* yp = yb + (size_t)(row0 + r) * a.y_pitch + t;
        const float bv = bias[r];
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (t + j < out_lim) yp[j] = yp[j] + a.sign * (acc[c][r][j] + bv);
      }
    }
  } else if constexpr (C::EPI == EPI_UPS8) {
    // packed row = co*8 + phase; thread owns one co, all 8 phases -> 32 contiguous outputs / chunk
    const int co = row0 >> 3;
    const float bv = a.bias[co];
    float* yb = a.y + (size_t)b * a.y_bs + (size_t)co * a.y_pitch;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int n = t0 + tb + 32 * c;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (n + j < out_lim) {
          float* yp = yb + (size_t)(n + j) * 8;
          *reinterpret_cast<float4*>(yp) =
              make_float4(acc[c][0][j] + bv, acc[c][1][j] + bv, acc[c][2][j] + bv, acc[c][3][j] + bv);
          *reinterpret_cast<float4*>(yp + 4) =
              make_float4(acc[c][4][j] + bv, acc[c][5][j] + bv, acc[c][6][j] + bv, acc[c][7][j] + bv);
        }
      }
    }
  } else if constexpr (C::EPI == EPI_UPS2) {
    // packed row = co*2 + phase; thread owns 4 co x 2 phases -> 8 contiguous outputs per co / chunk
    const int co0 = row0 >> 1;
    float* yb = a.y + (size_t)b * a.y_bs;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      const int n = t0 + tb + 32 * c;
      if (n >= out_lim) continue;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float bv = a.bias[co0 + i];
        float* yp = yb + (size_t)(co0 + i) * a.y_pitch + (size_t)n * 2;
        if (n + 3 < out_lim) {
          *reinterpret_cast<float4*>(yp) = make_float4(acc[c][2 * i][0] + bv, acc[c][2 * i + 1][0] + bv,
                                                       acc[c][2 * i][1] + bv, acc[c][2 * i + 1][1] + bv);
          *reinterpret_cast<float4*>(yp + 4) = make_float4(acc[c][2 * i][2] + bv, acc[c][2 * i + 1][2] + bv,
                                                           acc[c][2 * i][3] + bv, acc[c][2 * i + 1][3] + bv);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (n + j < out_lim) {
              yp[2 * j] = acc[c][2 * i][j] + bv;
              yp[2 * j + 1] = acc[c][2 * i + 1][j] + bv;
            }
        }
      }
    }
  }
}

// host-side launcher for one configuration
template <class C>
struct ConvLaunch {
  static cudaError_t prepare() {
    return cudaFuncSetAttribute(conv1d_f32<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM_BYTES);
  }
  static cudaError_t launch(const ConvArgs& a, int t_len, int row_tiles, int B, cudaStream_t st) {
    dim3 grid((t_len + C::T_T - 1) / C::T_T, row_tiles, B);
    conv1d_f32<C><<<grid, C::THREADS, C::SMEM_BYTES, st>>>(a);
    return cudaGetLastError();
  }
};

}  // namespace ovc
