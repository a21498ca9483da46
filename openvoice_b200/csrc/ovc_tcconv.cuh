// ovc_tcconv.cuh -- split-precision (3xFP16) tensor-core Conv1d for the generator / WaveNet convs.
//
//   Y[t, n] = (bias[n] + sum_{tap, c} W[n, c, tap] * lrelu(X[t + (tap - (K-1)/2) * DIL, c]) [+ R[t, n]] [+ Y_old[t, n]]) * scale
//
// Channels-last fp32 activations X[b][t][C] (time-major rows; fp16 in precision mode 3, tcconv_kernel<TN, true, true>).  Every operand is split x = hi + lo / 2^11 with
// hi = fp16(x), lo = fp16((x - hi) * 2^11) (22 mantissa bits, ovc_tc.cuh) and every product is evaluated as
// a_hi*b_hi + (a_lo*b_hi + a_hi*b_lo) / 2^11 by tcgen05.mma.kind::f16 with fp32 accumulation in TMEM: the hi*hi
// products in one accumulator, the two cross terms in a second one ("low-order accumulator"), joined in the
// epilogue.  The two accumulators of a tile sit side by side in TMEM and a weight slot holds [b_hi ; b_lo] as ONE
// 2*TN-row operand, so a_hi * [b_hi ; b_lo]^T is a single MMA of width 2*TN (both accumulators at once) and
// a_lo * b_hi^T a second one of width TN: two A-operand reads per k-step instead of three (SS-mode MMAs of the
// narrow layers are bound by shared-memory operand reads, 128 B/clk).  Besides carrying the 2^-11 scale, the second accumulator keeps the tensor core's truncating adds
// (tools/tc_acc_test.cu) away from the long hi*hi sum.  Error ~1e-6 per conv, i.e. fp32-grade
// (tools/tc_f16_test.cu); fp16 MMAs run at twice the TF32 rate on half the operand bytes.
//
// K-major, no-swizzle operand tiles (see ovc_tc.cuh): a convolution tap is a 16-byte-per-row shift of the A
// descriptor's start address, so all taps (any dilation) read ONE staged halo tile.  Two kernels:
//   tcconv_kernel<TN>        TN = 128 / 64 / 32 output columns, persistent: one CTA per SM walks the (utterance, tile)
//                            list, activations staged by TMA, epilogue of tile i under the MMAs of tile i+1
//   tcconv_wide_kernel       TN = 128, one 128-step tile per CTA, two CTAs per SM (the generator's first stage at k >= 7)
#pragma once
#include <cuda.h>   // CUtensorMap (the driver entry point that encodes it is resolved at run time, ovc_lib.cu)

#include "ovc_conv.cuh"
#include "ovc_tc.cuh"

namespace ovc {

struct TcConvArgs {
  const float* x; long long x_bs;     // [B][Lpitch][Cin]
  const uint16_t* w;                   // packed fp16 [n_tile][Cin/16][K][2 (8-channel column block)][hi|lo][TN][8]
  const float* bias; long long bias_bs; // [Ntot] (+ b * bias_bs: per-utterance speaker-conditioning bias of the WN gate)
  float* y; long long y_bs; int y_ld;  // [B][Lpitch][y_ld]
  const float* r;                      // residual, same geometry as y (nullable)
  float* s; long long s_bs;            // EPI 2: skip accumulator [B][Lpitch][y_ld]
  int epi;                             // 0 linear (bias, residual, accumulate, scale) | 1 WN gate | 2 WN res/skip
  int split; int first;                // EPI 2: columns < split update y (x += rs), the rest go to s[col - split] (= / +=)
  const long long* lens; int tmax; int mul;   // valid steps = min(tmax, lens[b]) * mul   (lens NULL -> tmax)
  const long long* lens_x; int has_lens_x;    // when set: the INPUT's own validity limit (generator conv_pre on a padded batch:
                                              // z_hat * y_mask is cut at the frame lengths, the output runs to tmax)
  int Cin; int Ntot; int K; int DIL;   // Ntot = output row width (C for a ResBlock conv, stride*Cout for a polyphase transposed conv)
  float slope; float scale; int accumulate;
  int passes;   // 3: split precision (a_hi*b_hi + a_lo*b_hi + a_hi*b_lo); 1: single-pass fp16 (11-bit operands, like cuDNN's TF32 default)
  int box_rows; int n_box;   // persistent kernel: an activation chunk arrives by tensor-map TMA as n_box boxes of box_rows x 32 channels
};

// one box of a [B][rows][Cin] fp32 tensor -> shared memory (128-byte swizzle), completion on an mbarrier
__device__ __forceinline__ void tma_tensor3d_g2s(void* dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
      : "memory");
}

// Programmatic dependent launch (launch_tc sets the stream-serialization attribute): the NEXT kernel's CTAs may start
// their prologue (barriers, TMEM, weight TMA) while this grid drains; a thread must pass pdl_wait() before it touches
// anything the PREVIOUS kernel wrote (or overwrites anything it read).
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

// item i of a staged chunk -> (row, 8-channel column block): 8 consecutive lanes take 8 consecutive rows of one
// column block, so the 16-byte operand stores of a quarter-warp are 128 contiguous bytes (conflict-free)
template <int NKC>
__device__ __forceinline__ void tc_item(int i, int& row, int& kc) {
  kc = (i >> 3) % NKC;
  row = (i / (8 * NKC)) * 8 + (i & 7);
}

// Storage type of the activations a kernel reads or writes: fp32, or fp16 (precision mode 3, the generator only).
// Two consecutive channels are loaded / stored as one float2 or half2 and the arithmetic is always fp32; an fp16 store
// rounds to nearest.
template <bool F16>
struct TcAct {
  using T = float;
};
template <>
struct TcAct<true> {
  using T = __half;
};
__device__ __forceinline__ float2 tc_ld2(const float* p) { return *reinterpret_cast<const float2*>(p); }
__device__ __forceinline__ float2 tc_ld2(const __half* p) { return __half22float2(*reinterpret_cast<const __half2*>(p)); }
__device__ __forceinline__ void tc_st2(float* p, float2 v) { *reinterpret_cast<float2*>(p) = v; }
__device__ __forceinline__ void tc_st2(__half* p, float2 v) { *reinterpret_cast<__half2*>(p) = __floats2half2_rn(v.x, v.y); }

// Epilogue of MMA tiles [mt_lo, mt_hi) x columns [c_lo, c_hi) of one CTA tile (MT x 128 steps x TN columns): TMEM ->
// registers -> fused ops -> global.  Warp w may read TMEM lanes [32*(w%4), +32); tile mt owns columns [2*mt*TN, +TN)
// (main accumulator) and the next TN (low-order accumulator).
// TMEM is read in the accumulator-fragment layout (tc::tmem_ld16x256_x4_issue): one block = 16 steps x 32 columns,
// four consecutive threads per 32-byte segment of an output row, so every global access of a warp is made of whole
// sectors (the thread-per-row layout moved 16 bytes per sector and spilled).  Operands with DRAM latency -- the
// residual of a ResBlock conv, the read-modify-write target of the WaveNet res/skip update -- are fetched one block
// ahead, and those of the first block BEFORE the wait on the accumulator barrier `bar`: they arrive under the MMAs.
// OUT16: y, r and the accumulate target are fp16 (half2 per thread and row, fp32 math, one rounding at the store); a
// quad then covers 16 bytes of a row per 8-column group, and groups g and g + 1 fill one 32-byte sector.
template <int TN, bool OUT16 = false>
__device__ __forceinline__ void tc_epilogue(const TcConvArgs& a, uint32_t acc, int b, int t0, int n0, int lim, int warp, int lane,
                                            int mt_lo, int mt_hi, int c_lo, int c_hi, uint64_t* bar, uint32_t parity) {
  using T = typename TcAct<OUT16>::T;
  const int lane_base = (warp & 3) * 32;
  const int rsub = lane >> 2, csub = (lane & 3) * 2;
  T* yb = reinterpret_cast<T*>(a.y) + (size_t)b * a.y_bs;
  const T* rb = a.r ? reinterpret_cast<const T*>(a.r) + (size_t)b * a.y_bs : nullptr;
  T* sb = a.s ? reinterpret_cast<T*>(a.s) + (size_t)b * a.s_bs : nullptr;
  const float* bias = a.bias + (size_t)b * a.bias_bs;
  const bool two = !OUT16 && a.passes == 3;   // the fp16-storage instantiations run one pass
  const int ncb = (c_hi - c_lo) >> 5;
  const int nblk = (mt_hi - mt_lo) * ncb * 2;

  // block k -> (MMA tile, 32-column group, 16-row half); rows a = first row of this thread, b = a + 8
  auto geom = [&](int k, int& mt, int& c0, int& row) {
    const int h = k & 1, q = k >> 1;
    mt = mt_lo + q / ncb;
    c0 = c_lo + (q % ncb) * 32;
    row = lane_base + 16 * h + rsub;
  };
  // where block k's read-modify-write / residual operand lives (nullptr: none)
  auto operand = [&](int c0, bool& add) -> const T* {
    add = true;
    if (OUT16 || a.epi == 0) return rb ? rb + n0 + c0 + csub : nullptr;
    if (a.epi == 2) {
      const int col = n0 + c0;
      const bool to_x = col < a.split;          // uniform per 32-column group (split is a multiple of 32)
      add = to_x || !a.first;
      return to_x ? yb + col + csub : sb + (col - a.split) + csub;
    }
    return nullptr;
  };
  auto prefetch = [&](int k, float2 (&q)[8]) {
    int mt, c0, row;
    geom(k, mt, c0, row);
    bool add;
    const T* src = operand(c0, add);
    const int ta = t0 + mt * 128 + row, tb = ta + 8;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      q[2 * g] = make_float2(0.f, 0.f);
      q[2 * g + 1] = make_float2(0.f, 0.f);
      if (src && add) {
        if (ta < lim) q[2 * g] = tc_ld2(src + (size_t)ta * a.y_ld + 8 * g);
        if (tb < lim) q[2 * g + 1] = tc_ld2(src + (size_t)tb * a.y_ld + 8 * g);
      }
    }
  };

  float2 rq[8];
  if (nblk > 0) prefetch(0, rq);
  mbar_wait(bar, parity);
  tc::fence_after();
#pragma unroll 1
  for (int k = 0; k < nblk; ++k) {
    int mt, c0, row;
    geom(k, mt, c0, row);
    const int ta = t0 + mt * 128 + row, tb = ta + 8;
    const bool oka = ta < lim, okb = tb < lim;
    const uint32_t taddr = acc + ((uint32_t)(lane_base + 16 * (k & 1)) << 16) + 2 * mt * TN + c0;
    uint32_t rm[16], rl[16];
    tc::tmem_ld16x256_x4_issue(taddr, rm);
    if (two) tc::tmem_ld16x256_x4_issue(taddr + TN, rl);
    // under the TMEM read: the next block's operand, this block's bias (and previous output when accumulating)
    float2 rn[8];
    if (k + 1 < nblk) {
      prefetch(k + 1, rn);
    } else {
#pragma unroll
      for (int g = 0; g < 8; ++g) rn[g] = make_float2(0.f, 0.f);
    }
    float2 bq[4], ya[4], yc[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) bq[g] = __ldg(reinterpret_cast<const float2*>(bias + n0 + c0 + 8 * g + csub));
    const bool accum = (OUT16 || a.epi == 0) && a.accumulate;
    if (accum) {
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        ya[g] = make_float2(0.f, 0.f);
        yc[g] = make_float2(0.f, 0.f);
        if (oka) ya[g] = tc_ld2(yb + (size_t)ta * a.y_ld + n0 + c0 + 8 * g + csub);
        if (okb) yc[g] = tc_ld2(yb + (size_t)tb * a.y_ld + n0 + c0 + 8 * g + csub);
      }
    }
    float v[16];
    if (two) {
      tc::tmem_ld_wait16x2(rm, rl);
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = fmaf(__uint_as_float(rl[i]), tc::kLoInv, __uint_as_float(rm[i]));
    } else {
      tc::tmem_ld_wait16(rm);
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(rm[i]);
    }
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      v[4 * g] += bq[g].x; v[4 * g + 1] += bq[g].y; v[4 * g + 2] += bq[g].x; v[4 * g + 3] += bq[g].y;
    }
    if (OUT16 || a.epi == 0) {   // an fp16 output has the linear epilogue only (launch_tc refuses the others)
      // ---- linear: bias, residual, MRF accumulate, scale (fp32 math; an fp16 output rounds once, at the store)
      T* ypa = yb + (size_t)ta * a.y_ld + n0 + c0 + csub;
      T* ypb = yb + (size_t)tb * a.y_ld + n0 + c0 + csub;
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        float2 oa = make_float2(v[4 * g] + rq[2 * g].x, v[4 * g + 1] + rq[2 * g].y);
        float2 ob = make_float2(v[4 * g + 2] + rq[2 * g + 1].x, v[4 * g + 3] + rq[2 * g + 1].y);
        if (accum) {
          oa.x = ya[g].x + oa.x; oa.y = ya[g].y + oa.y;
          ob.x = yc[g].x + ob.x; ob.y = yc[g].y + ob.y;
        }
        if (a.scale != 1.f) { oa.x *= a.scale; oa.y *= a.scale; ob.x *= a.scale; ob.y *= a.scale; }
        if (oka) tc_st2(ypa + 8 * g, oa);
        if (okb) tc_st2(ypb + 8 * g, ob);
      }
    } else if (a.epi == 1) {
      // ---- WaveNet gate (modules.py:185-210): columns [0,16) of the group are the tanh inputs of 16 channels,
      // [16,32) their sigmoid partners -> 16 output channels at column (n0 + c0) / 2
      T* ypa = yb + (size_t)ta * a.y_ld + ((n0 + c0) >> 1) + csub;
      T* ypb = yb + (size_t)tb * a.y_ld + ((n0 + c0) >> 1) + csub;
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        const float2 oa = make_float2(tanhf(v[4 * g]) * sigmoidf_acc(v[4 * (g + 2)]),
                                      tanhf(v[4 * g + 1]) * sigmoidf_acc(v[4 * (g + 2) + 1]));
        const float2 ob = make_float2(tanhf(v[4 * g + 2]) * sigmoidf_acc(v[4 * (g + 2) + 2]),
                                      tanhf(v[4 * g + 3]) * sigmoidf_acc(v[4 * (g + 2) + 3]));
        if (oka) tc_st2(ypa + 8 * g, oa);
        if (okb) tc_st2(ypb + 8 * g, ob);
      }
    } else {
      // ---- WaveNet res/skip: columns < split update x in place (x += res), the rest go to the skip sum (= / +=)
      bool add;
      T* dst = const_cast<T*>(operand(c0, add));
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const float2 oa = make_float2(rq[2 * g].x + v[4 * g], rq[2 * g].y + v[4 * g + 1]);
        const float2 ob = make_float2(rq[2 * g + 1].x + v[4 * g + 2], rq[2 * g + 1].y + v[4 * g + 3]);
        if (oka) tc_st2(dst + (size_t)ta * a.y_ld + 8 * g, oa);
        if (okb) tc_st2(dst + (size_t)tb * a.y_ld + 8 * g, ob);
      }
    }
#pragma unroll
    for (int g = 0; g < 8; ++g) rq[g] = rn[g];
  }
}

// The MMAs of one (k-step, tap) of one 128-row MMA tile against weight slot b = [b_hi ; b_lo] (2 x TN rows), the A
// tile's lo parts a_lo16 16-byte units after its hi parts.  Three passes: [main | low] (+)= a_hi * [b_hi ; b_lo]^T,
// low += a_lo * b_hi^T; one pass: main (+)= a_hi * b_hi^T.  For one thread: the issuing warp runs its loop converged
// and calls this under tc::elect_one() (ovc_tc.cuh: a divergent issuer costs a replay sequence per MMA).
template <int TN>
__device__ __forceinline__ void tc_mma_step(uint32_t acc, uint64_t a_hi, uint32_t a_lo16, uint64_t b, bool three, bool accumulate) {
  constexpr uint32_t idesc1 = tc::make_idesc_f16(128, TN), idesc2 = tc::make_idesc_f16(128, 2 * TN);
  if (three) {
    tc::mma_f16(acc, a_hi, b, idesc2, accumulate);
    tc::mma_f16(acc + TN, a_hi + a_lo16, b, idesc1, true);
  } else {
    tc::mma_f16(acc, a_hi, b, idesc1, accumulate);
  }
}

// A raw fp32 stage of rows x 32 channels (row r = step t_first + r), 128-byte swizzled: 16-byte piece c of row r sits
// at r * 128 + ((c ^ (r & 7)) << 4) -> leaky-relu -> hi/lo operand tile of row pitch ROWS (column block kc of row r at
// (kc * ROWS + r) * 16, the lo parts after the 4 hi column blocks).  Rows outside [0, lim) become zeros: zero padding,
// x_mask and the ragged batch in one rule.  Item i = (row i / 4, column block i % 4), NT threads, thread pt.  Two items
// per iteration: both pairs of shared-memory loads are in flight before the first conversion (one item at a time left
// the LDS latency exposed: a single warp per scheduler runs this role).
template <int ROWS, int NT>
__device__ __forceinline__ void tc_convert_raw(const unsigned char* raw, unsigned char* ah, int pt, int items, int t_first, int lim,
                                               float slope) {
  unsigned char* al = ah + 4 * ROWS * 16;
  auto fetch = [&](int i, float4& v0, float4& v1) {
    const int row = i >> 2, kc = i & 3;
    const int t = t_first + row;
    v0 = make_float4(0.f, 0.f, 0.f, 0.f);
    v1 = v0;
    if (i < items && t >= 0 && t < lim) {
      const unsigned char* rr = raw + row * 128;
      v0 = *reinterpret_cast<const float4*>(rr + (((2 * kc) ^ (row & 7)) << 4));
      v1 = *reinterpret_cast<const float4*>(rr + (((2 * kc + 1) ^ (row & 7)) << 4));
    }
  };
  auto emit = [&](int i, const float4& v0, const float4& v1) {
    if (i >= items) return;
    const int row = i >> 2, kc = i & 3;
    uint4 hi, lo;
    tc::split_f16x8(v0, v1, slope, hi, lo);
    *reinterpret_cast<uint4*>(ah + (kc * ROWS + row) * 16) = hi;
    *reinterpret_cast<uint4*>(al + (kc * ROWS + row) * 16) = lo;
  };
  for (int i = pt; i < items; i += 2 * NT) {
    float4 a0, a1, b0, b1;
    fetch(i, a0, a1);
    fetch(i + NT, b0, b1);
    emit(i, a0, a1);
    emit(i + NT, b0, b1);
  }
}

// The fp16 counterpart (precision mode 3): a raw fp16 stage of rows x 32 channels, 64 bytes per row, unswizzled ->
// leaky-relu in fp32 -> fp16 (round to nearest) -> the hi operand tile only (one pass: there is no lo tile).  Item i =
// (row i / 4, column block i % 4) is one 16-byte piece, so the 8 lanes of a quarter-warp read two whole rows, 128
// contiguous bytes: conflict-free without a swizzle.  Rows outside [0, lim) become zeros, as above.
template <int ROWS, int NT>
__device__ __forceinline__ void tc_convert_raw16(const unsigned char* raw, unsigned char* ah, int pt, int items, int t_first, int lim,
                                                 float slope) {
  auto fetch = [&](int i, uint4& v) {
    const int row = i >> 2, kc = i & 3;
    const int t = t_first + row;
    v = make_uint4(0u, 0u, 0u, 0u);
    if (i < items && t >= 0 && t < lim) v = *reinterpret_cast<const uint4*>(raw + row * 64 + kc * 16);
  };
  auto emit = [&](int i, uint4 v) {
    if (i >= items) return;
    const int row = i >> 2, kc = i & 3;
    uint32_t h[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float2 f = __half22float2(*reinterpret_cast<const __half2*>(&h[k]));
      f.x = fmaxf(f.x, f.x * slope);   // leaky_relu, as in tc::split_f16x8
      f.y = fmaxf(f.y, f.y * slope);
      const __half2 r = __floats2half2_rn(f.x, f.y);
      h[k] = *reinterpret_cast<const uint32_t*>(&r);
    }
    *reinterpret_cast<uint4*>(ah + (kc * ROWS + row) * 16) = make_uint4(h[0], h[1], h[2], h[3]);
  };
  for (int i = pt; i < items; i += 2 * NT) {
    uint4 a, b;
    fetch(i, a);
    fetch(i + NT, b);
    emit(i, a);
    emit(i + NT, b);
  }
}

// Tile `tile` of a persistent kernel's (utterance, tile) list, `steps` output steps per tile: utterance b, first step t0,
// valid steps lim = min(tmax, lens[b]) * mul (lens NULL: tmax * mul) and the input's own limit lim_x (the same from
// lens_x; lens_x NULL: lim).  A tile with t0 >= lim lies past its utterance's end: every role skips it.
struct TcTile {
  int b, t0, lim, lim_x;
};
__device__ __forceinline__ TcTile tc_tile(int tile, int n_tt, int steps, const long long* lens, const long long* lens_x, int tmax,
                                          int mul) {
  TcTile t;
  t.b = tile / n_tt;
  t.t0 = (tile % n_tt) * steps;
  t.lim = (lens ? (int)min((long long)tmax, lens[t.b]) : tmax) * mul;
  t.lim_x = lens_x ? (int)min((long long)tmax, lens_x[t.b]) * mul : t.lim;
  return t;
}

// n weight slots of SLOT bytes, resident for the whole launch: one thread copies them from `src` into slots [0, n) of
// `ring` (completion on bars[0, n)) and waits for them.  A CTA whose tiles all lie past their utterances never waits on
// these copies otherwise, and they must have landed before it exits (its shared memory may go to the next kernel's CTA).
template <int SLOT>
__device__ __forceinline__ void tc_load_resident(unsigned char* ring, uint64_t* bars, const void* src, int n) {
  const unsigned char* s = reinterpret_cast<const unsigned char*>(src);
  for (int it = 0; it < n; ++it) {
    mbar_expect_tx(&bars[it], SLOT);
    tma_bulk_g2s(ring + it * SLOT, s + (size_t)it * SLOT, SLOT, &bars[it]);
  }
  for (int it = 0; it < n; ++it) mbar_wait(&bars[it], 0u);
}

// ---------------------------------------------------------------------------------------------------------
// tcconv_wide_kernel: TN = 128 output columns, one 128-step tile per CTA: 256 TMEM columns and ~109 KB of shared
// memory per CTA -> TWO CTAs per SM, so one CTA's prologue / epilogue overlaps the other's MMAs (the layer's weights
// are re-streamed per 128 steps).
// (A 2-CTA-cluster variant that multicast the weight stream was measured in round 2: no faster, and wrong results
// whenever both CTAs of a cluster were active -- removed.)
// Warp roles: warp 0 TMA weight producer; warp 1 one MMA-issuing thread; warps 2..5 A producers (cp.async raw rows
// RAWD chunks ahead -> lrelu -> hi/lo fp16 split -> operand layout), then epilogue.
// ---------------------------------------------------------------------------------------------------------
struct TcwCfg {
  static constexpr int TN = 128;
  static constexpr int KCH = 16, NKC = KCH / 8, KS = KCH / 16;    // channels per A stage
  static constexpr int THREADS = 192;
  static constexpr int ROWS = 128 + 64;                           // staged rows per A buffer (tile + 2*25 halo, padded)
  static constexpr int NABUF = 2;                                 // converted A stages
  static constexpr int RAWD = 2, NST = RAWD + 1;                  // raw fp32 landing stages in flight ahead
  static constexpr int SLOTS = 6;                                 // weight ring depth
  static constexpr int A_BUF_BYTES = 2 * NKC * ROWS * 16;         // [hi|lo][column block][row][8 halfs]
  static constexpr int SLOT_BYTES = 2 * 2 * TN * 16;              // [column block][hi|lo][n][8 halfs]
  static constexpr int RAW_BYTES = ROWS * KCH * 4;
  static constexpr size_t SMEM_BYTES = 512 + NABUF * A_BUF_BYTES + SLOTS * SLOT_BYTES + NST * RAW_BYTES;
  static constexpr uint32_t TMEM_COLS = 2 * TN;                   // main + low-order accumulators
};

__global__ void __launch_bounds__(TcwCfg::THREADS, 2) tcconv_wide_kernel(const TcConvArgs a) {
  using Cfg = TcwCfg;
  constexpr int TN = Cfg::TN, NABUF = Cfg::NABUF, SLOTS = Cfg::SLOTS, ROWS = Cfg::ROWS, NKC = Cfg::NKC;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
  uint64_t* a_full = bars, *a_empty = bars + NABUF, *b_full = bars + 2 * NABUF, *b_empty = b_full + SLOTS,
            *acc_full = b_empty + SLOTS;
  static_assert((2 * NABUF + 2 * SLOTS + 1) * 8 + 8 <= 512, "barrier area");
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);
  unsigned char* abuf = smem_raw + 512;
  unsigned char* bring = abuf + NABUF * Cfg::A_BUF_BYTES;
  unsigned char* raw = bring + SLOTS * Cfg::SLOT_BYTES;

  const int b = blockIdx.z;
  const int t0 = blockIdx.x * 128;
  const int n0 = blockIdx.y * TN;
  const int lim = (a.lens ? (int)min((long long)a.tmax, a.lens[b]) : a.tmax) * a.mul;
  const int lim_x = a.has_lens_x ? (int)min((long long)a.tmax, a.lens_x[b]) * a.mul : lim;
  if (t0 >= lim) return;   // the tile lies past the utterance

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // provably warp-uniform: role code may use uniform registers
  const int H = (a.K - 1) / 2 * a.DIL;
  const int nq = a.Cin / Cfg::KCH;            // A chunks
  const int n_slots = (a.Cin / 16) * a.K;

  if (tid == 0) {
    for (int i = 0; i < NABUF; ++i) { mbar_init(&a_full[i], 128); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < SLOTS; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
    mbar_init(acc_full, 1);
    fence_mbar_init();
  }
  if (warp == 1) tc::tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  tc::fence_before();
  __syncthreads();
  tc::fence_after();
  const uint32_t tmem_d = *tmem_slot;
  pdl_launch_dependents();
  if (warp != 0) pdl_wait();   // warp 0 only streams the (constant) weights: it may run ahead of the previous kernel's end

  if (warp == 0) {
    // ------------------------------------------------------------ weight producer (TMA bulk)
    if (lane == 0) {
      const unsigned char* wp = reinterpret_cast<const unsigned char*>(a.w) + (size_t)blockIdx.y * n_slots * Cfg::SLOT_BYTES;
      constexpr uint32_t BYTES = Cfg::SLOT_BYTES;
      int slot = 0;
      uint32_t phase = 1;   // the first pass over the ring finds every slot free
      for (int it = 0; it < n_slots; ++it) {
        mbar_wait(&b_empty[slot], phase);
        mbar_expect_tx(&b_full[slot], BYTES);
        tma_bulk_g2s(bring + slot * Cfg::SLOT_BYTES, wp, BYTES, &b_full[slot]);
        wp += Cfg::SLOT_BYTES;
        if (++slot == SLOTS) { slot = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (one elected thread)
    // The whole warp runs the loop converged and only the tcgen05 instructions are predicated on elect.sync: the
    // descriptors then live in uniform registers and advance by plain adds (they differ only in their 14-bit
    // start-address field).  [A divergent `if (lane == 0)` around the loop made ptxas wrap every MMA in an
    // ELECT / R2UR / BRA.U.ANY replay sequence: ~60 dependent instructions per MMA pair, 35 % tensor-pipe activity.]
    {
      constexpr uint32_t LBO_A = ROWS * 16, LBO_B = 2 * TN * 16, SBO = 128;
      constexpr uint32_t A_LO16 = (NKC * ROWS * 16) >> 4;        // hi -> lo inside an A buffer, in 16-byte units
      constexpr uint32_t SLOT16 = Cfg::SLOT_BYTES >> 4;
      const uint64_t a_proto = tc::make_desc(0, LBO_A, SBO), b_proto = tc::make_desc(0, LBO_B, SBO);
      const uint64_t b_ring = b_proto + (tc::smem_addr(bring) >> 4);
      const uint32_t dil = (uint32_t)a.DIL;
      const bool three = a.passes == 3;
      int slot = 0;
      uint32_t bphase = 0;
      bool first = true;
      for (int q = 0; q < nq; ++q) {
        const int buf = q % NABUF;
        mbar_wait(&a_full[buf], (q / NABUF) & 1);
        tc::fence_after();
        for (int j = 0; j < Cfg::KS; ++j) {
          uint64_t a_cur = a_proto + ((tc::smem_addr(abuf + buf * Cfg::A_BUF_BYTES) + 2 * j * LBO_A) >> 4);
          for (int tap = 0; tap < a.K; ++tap) {
            mbar_wait(&b_full[slot], bphase);
            tc::fence_after();
            const uint64_t b_slot = b_ring + (uint32_t)slot * SLOT16;
            // output step (t0 + i) reads staged row (i + tap*DIL): the halo tile starts at t0 - H
            if (tc::elect_one()) {
              tc_mma_step<TN>(tmem_d, a_cur, A_LO16, b_slot, three, !first);
              tc::mma_commit(&b_empty[slot]);       // slot reusable once these MMAs have read it
            }
            __syncwarp();
            first = false;
            a_cur += dil;
            if (++slot == SLOTS) { slot = 0; bphase ^= 1; }
          }
        }
        if (tc::elect_one()) tc::mma_commit(&a_empty[buf]);
        __syncwarp();
      }
      if (tc::elect_one()) tc::mma_commit(acc_full);
      __syncwarp();
    }
  } else if (warp >= 2 && warp <= 5) {
    // ------------------------------------------------------------ A producers, then epilogue
    const int pt = tid - 64;                                   // 0..127
    const float* xb = a.x + (size_t)b * a.x_bs;
    const int rows8 = (128 + 2 * H + 7) & ~7;
    constexpr int NP = Cfg::KCH / 4;                           // 16-byte pieces per raw row
    const int pieces = rows8 * NP, items = rows8 * NKC;
    // raw fp32 rows land by cp.async (zero-filled outside [0, lim)), fully coalesced, RAWD chunks ahead; piece p of
    // row r sits at 16-byte slot r*NP + (p ^ ((r >> 1) & 3)) so the conversion's row-strided reads are conflict-free
    auto stage = [&](int q) {
      unsigned char* dst = raw + (q % Cfg::NST) * Cfg::RAW_BYTES;
      for (int i = pt; i < pieces; i += 128) {
        const int row = i / NP, p = i % NP;
        const int t = t0 - H + row;
        const bool ok = (t >= 0 && t < lim_x);
        const float* src = ok ? xb + (size_t)t * a.Cin + q * Cfg::KCH + p * 4 : xb;
        cp_async16_zfill(dst + (row * NP + (p ^ ((row >> 1) & 3))) * 16, src, ok ? 16 : 0);
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    for (int q = 0; q < Cfg::RAWD; ++q) {
      if (q < nq) stage(q);
      else asm volatile("cp.async.commit_group;" ::: "memory");
    }
    for (int q = 0; q < nq; ++q) {
      asm volatile("cp.async.wait_group %0;" ::"n"(Cfg::RAWD - 1) : "memory");   // this thread's pieces of chunk q landed
      named_bar_sync(1, 128);   // ... everybody's did, and everybody is done reading the stage refilled next
      if (q + Cfg::RAWD < nq) stage(q + Cfg::RAWD);
      else asm volatile("cp.async.commit_group;" ::: "memory");                   // keep the group count uniform
      const int buf = q % NABUF;
      mbar_wait(&a_empty[buf], ((q / NABUF) & 1) ^ 1);
      unsigned char* ah = abuf + buf * Cfg::A_BUF_BYTES;
      unsigned char* al = ah + NKC * ROWS * 16;
      const unsigned char* src = raw + (q % Cfg::NST) * Cfg::RAW_BYTES;
      for (int i = pt; i < items; i += 128) {
        int row, kc;
        tc_item<NKC>(i, row, kc);
        const int sw = (row >> 1) & 3;
        const float4 v0 = *reinterpret_cast<const float4*>(src + (row * NP + ((2 * kc) ^ sw)) * 16);
        const float4 v1 = *reinterpret_cast<const float4*>(src + (row * NP + ((2 * kc + 1) ^ sw)) * 16);
        uint4 hi, lo;
        tc::split_f16x8(v0, v1, a.slope, hi, lo);
        *reinterpret_cast<uint4*>(ah + (kc * ROWS + row) * 16) = hi;
        *reinterpret_cast<uint4*>(al + (kc * ROWS + row) * 16) = lo;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> tensor-core (async) proxy
      mbar_arrive(&a_full[buf]);
    }
    // epilogue: warp w may read TMEM lanes [32*(w%4), +32)
    tc_epilogue<TN>(a, tmem_d, b, t0, n0, lim, warp, lane, 0, 1, 0, TN, acc_full, 0);
  }
  tc::fence_before();
  __syncthreads();
  if (warp == 1) tc::tmem_dealloc(tmem_d, Cfg::TMEM_COLS);
}

// ---------------------------------------------------------------------------------------------------------
// tcconv_kernel<TN>: persistent split-precision conv, TN = 128 / 64 / 32 output columns per CTA.
// One CTA per SM loops over tiles (TN = 128: 128 steps, else 256): barriers / TMEM live for the whole launch, the
// layer's weights stay resident in shared memory when they fit (C = 32: <= 44 KB; C = 64, k = 3: 48 KB; otherwise a
// ring streams them per tile), and every stage runs ahead across tile boundaries:
//   warp 15     activation TMA: a chunk of a halo tile = rows x 32 channels of the channels-last tensor is
//               ONE tensor-map box (two when it has more than 256 rows): cp.async.bulk.tensor lands it in a raw fp32
//               stage, 128-byte swizzled, NRAW chunks ahead, rows before the tensor's start zero-filled by the copy
//               engine -- the copy engine, not registers, holds the bytes in flight (the narrow layers are HBM-bound:
//               a whole tile must be in flight per SM to cover the latency).  [Measured: one 128-byte bulk copy per
//               row instead costs ~55 cycles of TMA issue each and caps the kernel at 1.1 TB/s.]
//   warps 3-6   (2-6 when TN = 128: its second MMA-issuer warp is free) converters: raw stage -> lrelu -> fp16 hi/lo
//               split -> operand layout (tc_convert_raw)
//   warp 0      weight TMA; warps 1-2 one MMA-issuing thread each (TN = 128: one)
//   warps 7-14  epilogue of tile i (second TMEM accumulator set) while the MMAs of tile i+1 run
// The raw stage's 128-byte swizzle and the operand tiles' ROWS = 2 (mod 8) column-block pitch make both sides of
// the conversion shared-memory bank-conflict free.
// ---------------------------------------------------------------------------------------------------------
constexpr int TCN_THREADS = 512;

template <int TN>
struct TcnCfg {
  static constexpr int MT = TN == 128 ? 1 : 2;                    // 2 sets x MT x (main + low-order) x TN <= 512 TMEM columns
  static constexpr int NISS = MT >= 2 ? 2 : 1;
  static constexpr int CONV_W0 = 1 + NISS;                        // first converter warp: with one MMA issuer (TN = 128) warp 2
  static constexpr int NCT = (7 - CONV_W0) * 32;                  // joins the converters (5 warps instead of 4)
  static constexpr int KCH = 32, NKC = KCH / 8, KS = KCH / 16;
  static constexpr int ROWS = MT * 128 + 66;                      // = 2 (mod 8)
  static constexpr int RAW_ROWS = MT == 1 ? 184 : 320;            // tile + 2 * 25 halo, rounded up to 8 (16 when two boxes)
  static constexpr int NABUF = 2;
  static constexpr int NRAW = TN == 128 ? 3 : 2;                  // raw fp32 chunk stages
  static constexpr int RAW_STAGE_BYTES = RAW_ROWS * 128;          // multiple of 1024: every stage keeps the swizzle phase
  static constexpr int RING = TN == 32 ? 22 : (TN == 64 ? 12 : 13);   // weight slots: 44 KB / 48 KB / 104 KB
  static constexpr int A_BUF_BYTES = 2 * NKC * ROWS * 16;
  static constexpr int SLOT_BYTES = 2 * 2 * TN * 16;
  static constexpr size_t SMEM_BYTES = 1024 + NABUF * A_BUF_BYTES + RING * SLOT_BYTES + 1024 + NRAW * RAW_STAGE_BYTES;
  static constexpr uint32_t TMEM_COLS = 2 * 2 * MT * TN;          // 512 (TN 128, 64) / 256 (TN 32)
};

// rows staged per chunk: the tile plus its halo, rounded so that one box (<= 256 rows) or two equal boxes of a
// multiple of 8 rows cover it
__host__ __device__ inline int tcn_rows(int mt, int H) {
  const int r = mt * 128 + 2 * H;
  return r <= 256 ? (r + 7) & ~7 : (r + 15) & ~15;
}

// IN16 / OUT16: the activations read / written are fp16 (precision mode 3).  An fp16 raw stage holds 64-byte rows in
// the same stage buffers (half of each is used), and these instantiations run one fp16 pass per conv.
template <int TN, bool IN16 = false, bool OUT16 = false>
__global__ void __launch_bounds__(TCN_THREADS, 1) tcconv_kernel(const TcConvArgs a, int n_tt, int total,
                                                                const __grid_constant__ CUtensorMap tmap) {
  using Cfg = TcnCfg<TN>;
  constexpr int MT = Cfg::MT, ROWS = Cfg::ROWS, NABUF = Cfg::NABUF, RING = Cfg::RING, NKC = Cfg::NKC, NRAW = Cfg::NRAW,
                NISS = Cfg::NISS, NCT = Cfg::NCT;
  constexpr uint32_t SET_COLS = 2 * MT * TN;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
  uint64_t* a_full = bars, *a_empty = bars + NABUF, *b_full = bars + 2 * NABUF, *b_empty = b_full + RING,
            *acc_full = b_empty + RING, *acc_empty = acc_full + 2, *raw_full = acc_empty + 2, *raw_empty = raw_full + NRAW;
  static_assert((2 * NABUF + 2 * RING + 4 + 2 * NRAW) * 8 + 8 <= 1024, "barrier area");
  static_assert(Cfg::SMEM_BYTES <= 232448, "shared memory budget");
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(raw_empty + NRAW);
  unsigned char* abuf = smem_raw + 1024;
  unsigned char* bring = abuf + NABUF * Cfg::A_BUF_BYTES;
  // raw stages: 1024-byte aligned in the shared window (the 128-byte swizzle is a function of address bits 4..9)
  unsigned char* raw = bring + RING * Cfg::SLOT_BYTES;
  raw += (1024u - (smem_u32(raw) & 1023u)) & 1023u;

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // provably warp-uniform: role code may use uniform registers
  const int n0 = blockIdx.y * TN;
  const int H = (a.K - 1) / 2 * a.DIL;
  const int rows8 = tcn_rows(MT, H);
  const int nq = a.Cin / Cfg::KCH;
  const int n_slots = (a.Cin / 16) * a.K;
  const bool resident = n_slots <= RING;
  const long long* lens_x = a.has_lens_x ? a.lens_x : nullptr;
  constexpr uint32_t BYTES = Cfg::SLOT_BYTES;

  if (tid == 0) {
    for (int i = 0; i < NABUF; ++i) { mbar_init(&a_full[i], NCT); mbar_init(&a_empty[i], NISS); }
    for (int i = 0; i < RING; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], NISS); }
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], NISS); mbar_init(&acc_empty[i], 8); }
    for (int i = 0; i < NRAW; ++i) { mbar_init(&raw_full[i], 1); mbar_init(&raw_empty[i], NCT); }
    fence_mbar_init();
  }
  if (warp == 1) tc::tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  tc::fence_before();
  __syncthreads();
  tc::fence_after();
  const uint32_t tmem_d = *tmem_slot;
  pdl_launch_dependents();
  if (warp != 0) pdl_wait();   // warp 0 only streams the (constant) weights: it may run ahead of the previous kernel's end

  // every role walks the same tile sequence
  if (warp == 0) {
    // ------------------------------------------------------------ weights
    if (lane == 0) {
      const unsigned char* wt = reinterpret_cast<const unsigned char*>(a.w) + (size_t)blockIdx.y * n_slots * Cfg::SLOT_BYTES;
      if (resident) {
        tc_load_resident<Cfg::SLOT_BYTES>(bring, b_full, wt, n_slots);
      } else {
        int slot = 0;
        uint32_t phase = 1;
        for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
          const TcTile tl = tc_tile(tile, n_tt, MT * 128, a.lens, lens_x, a.tmax, a.mul);
          if (tl.t0 >= tl.lim) continue;
          for (int it = 0; it < n_slots; ++it) {
            mbar_wait(&b_empty[slot], phase);
            mbar_expect_tx(&b_full[slot], BYTES);
            tma_bulk_g2s(bring + slot * Cfg::SLOT_BYTES, wt + (size_t)it * Cfg::SLOT_BYTES, BYTES, &b_full[slot]);
            if (++slot == RING) { slot = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 15) {
    // ------------------------------------------------------------ activation chunks by tensor-map TMA
    if (lane == 0) {
      int st = 0;
      uint32_t phase = 1;   // the first pass finds every raw stage free
      const uint32_t box_bytes = (uint32_t)a.box_rows * (IN16 ? 64u : 128u);
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const TcTile tl = tc_tile(tile, n_tt, MT * 128, a.lens, lens_x, a.tmax, a.mul);
        if (tl.t0 >= tl.lim) continue;
        for (int q = 0; q < nq; ++q) {
          mbar_wait(&raw_empty[st], phase);
          mbar_expect_tx(&raw_full[st], box_bytes * (uint32_t)a.n_box);
          unsigned char* dst = raw + st * Cfg::RAW_STAGE_BYTES;
          for (int i = 0; i < a.n_box; ++i)   // coordinates: channel, row (may be negative: zero-filled), utterance
            tma_tensor3d_g2s(dst + i * box_bytes, &tmap, q * Cfg::KCH, tl.t0 - H + i * a.box_rows, tl.b, &raw_full[st]);
          if (++st == NRAW) { st = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1 || (NISS == 2 && warp == 2)) {
    // ------------------------------------------------------------ MMA issuers (one elected thread per warp, converged loop)
    {
      static_assert(MT == NISS, "one MMA tile per issuer");
      const int mt = warp - 1;
      constexpr uint32_t LBO_A = ROWS * 16, LBO_B = 2 * TN * 16, SBO = 128;
      constexpr uint32_t A_LO16 = (NKC * ROWS * 16) >> 4, SLOT16 = Cfg::SLOT_BYTES >> 4;
      const uint64_t a_proto = tc::make_desc(0, LBO_A, SBO) + mt * 128, b_proto = tc::make_desc(0, LBO_B, SBO);
      const uint64_t b_ring = b_proto + (tc::smem_addr(bring) >> 4);
      const uint32_t dil = (uint32_t)a.DIL;
      const bool three = !(IN16 || OUT16) && a.passes == 3;
      int slot = 0, buf = 0, n = 0;
      uint32_t bphase = 0, aphase = 0;
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const TcTile tl = tc_tile(tile, n_tt, MT * 128, a.lens, lens_x, a.tmax, a.mul);
        if (tl.t0 >= tl.lim) continue;
        const int set = n & 1;
        mbar_wait(&acc_empty[set], ((n >> 1) & 1) ^ 1);   // the epilogue has drained this accumulator set
        tc::fence_after();
        const uint32_t acc = tmem_d + set * SET_COLS + 2 * mt * TN;
        bool first = true;
        if (resident) slot = 0;
        for (int q = 0; q < nq; ++q) {
          mbar_wait(&a_full[buf], aphase);
          tc::fence_after();
          for (int j = 0; j < Cfg::KS; ++j) {
            uint64_t a_cur = a_proto + ((tc::smem_addr(abuf + buf * Cfg::A_BUF_BYTES) + 2 * j * LBO_A) >> 4);
            for (int tap = 0; tap < a.K; ++tap) {
              if (!resident || n == 0) {
                mbar_wait(&b_full[slot], resident ? 0u : bphase);
                tc::fence_after();
              }
              const uint64_t b_slot = b_ring + (uint32_t)slot * SLOT16;
              if (tc::elect_one()) {
                tc_mma_step<TN>(acc, a_cur, A_LO16, b_slot, three, !first);
                if (!resident) tc::mma_commit(&b_empty[slot]);
              }
              __syncwarp();
              first = false;
              a_cur += dil;
              if (++slot == RING) { slot = 0; bphase ^= 1; }
            }
          }
          if (tc::elect_one()) tc::mma_commit(&a_empty[buf]);
          __syncwarp();
          if (++buf == NABUF) { buf = 0; aphase ^= 1; }
        }
        if (tc::elect_one()) tc::mma_commit(&acc_full[set]);
        __syncwarp();
        ++n;
      }
    }
  } else if (warp >= Cfg::CONV_W0 && warp <= 6) {
    // ------------------------------------------------------------ converters (run ahead across tiles)
    const int pt = tid - 32 * Cfg::CONV_W0;
    const int items = rows8 * NKC;            // item i = (row i / 4, column block i % 4): 32 bytes of one row
    int buf = 0, st = 0;
    uint32_t ephase = 1, rphase = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
      const TcTile tl = tc_tile(tile, n_tt, MT * 128, a.lens, lens_x, a.tmax, a.mul);
      if (tl.t0 >= tl.lim) continue;
      for (int q = 0; q < nq; ++q) {
        mbar_wait(&raw_full[st], rphase);
        mbar_wait(&a_empty[buf], ephase);
        if constexpr (IN16)
          tc_convert_raw16<ROWS, NCT>(raw + st * Cfg::RAW_STAGE_BYTES, abuf + buf * Cfg::A_BUF_BYTES, pt, items, tl.t0 - H, tl.lim_x,
                                      a.slope);
        else
          tc_convert_raw<ROWS, NCT>(raw + st * Cfg::RAW_STAGE_BYTES, abuf + buf * Cfg::A_BUF_BYTES, pt, items, tl.t0 - H, tl.lim_x,
                                    a.slope);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_arrive(&a_full[buf]);
        if (++buf == NABUF) { buf = 0; ephase ^= 1; }
        mbar_arrive(&raw_empty[st]);          // this thread has read everything it needs from the raw stage
        if (++st == NRAW) { st = 0; rphase ^= 1; }
      }
    }
  } else if (warp >= 7 && warp <= 14) {
    // ------------------------------------------------------------ epilogue (overlaps the next tile's MMAs)
    // each warp covers the TMEM lane quadrant warp % 4; warps 7..10 / 11..14 split the MMA tiles (MT = 2) or the
    // columns (MT = 1) of the CTA tile between them
    const int half = (warp - 7) >> 2;
    const int mt_lo = MT == 2 ? half : 0, mt_hi = MT == 2 ? half + 1 : 1;
    const int c_lo = MT == 2 ? 0 : half * (TN / 2), c_hi = MT == 2 ? TN : c_lo + TN / 2;
    int n = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
      const TcTile tl = tc_tile(tile, n_tt, MT * 128, a.lens, lens_x, a.tmax, a.mul);
      if (tl.t0 >= tl.lim) continue;
      const int set = n & 1;
      tc_epilogue<TN, OUT16>(a, tmem_d + set * SET_COLS, tl.b, tl.t0, n0, tl.lim, warp, lane, mt_lo, mt_hi, c_lo, c_hi, &acc_full[set],
                      (n >> 1) & 1);
      tc::fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[set]);
      ++n;
    }
  }
  tc::fence_before();
  __syncthreads();
  if (warp == 1) tc::tmem_dealloc(tmem_d, Cfg::TMEM_COLS);
}

// four consecutive channels of an fp32 or fp16 activation row
__device__ __forceinline__ float4 ld_f4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld_f4(const __half* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}

// conv_post on channels-last input (fp32, or fp16 in precision mode 3): y[b, t] = tanh(sum_{k<7, ci<C} w[ci, k] * lrelu_0.01(x[b, t+k-3, ci]))
// (models.py:287-289).  HBM-bound (132 B per sample): a CTA stages 256+6 rows with coalesced 16-byte loads into a
// transposed, conflict-free shared tile (leaky_relu applied once), then one thread per output sample.
template <int C, class T = float>
__global__ void __launch_bounds__(256) conv_post_cl_kernel(const T* __restrict__ x, long long x_bs,
                                                           const float* __restrict__ w, float* __restrict__ y,
                                                           long long y_bs, int y_len, const long long* lens, int tmax,
                                                           int mul) {
  constexpr int TB = 256, ROWS = TB + 6, LD = ROWS + 3;   // LD odd: conflict-free transposed stores
  __shared__ float ws[7][C];
  __shared__ float xs[C][LD];
  for (int i = threadIdx.x; i < C * 7; i += blockDim.x) ws[i % 7][i / 7] = w[i];
  const int b = blockIdx.y;
  const int lim = (lens ? (int)min((long long)tmax, lens[b]) : tmax) * mul;
  const int t0 = blockIdx.x * TB;
  const T* xb = x + (size_t)b * x_bs;
  for (int idx = threadIdx.x; idx < ROWS * (C / 4); idx += blockDim.x) {
    const int row = idx / (C / 4), q = idx % (C / 4);
    const int tt = t0 - 3 + row;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tt >= 0 && tt < lim) v = ld_f4(xb + (size_t)tt * C + 4 * q);
    xs[4 * q + 0][row] = v.x > 0.f ? v.x : 0.01f * v.x;
    xs[4 * q + 1][row] = v.y > 0.f ? v.y : 0.01f * v.y;
    xs[4 * q + 2][row] = v.z > 0.f ? v.z : 0.01f * v.z;
    xs[4 * q + 3][row] = v.w > 0.f ? v.w : 0.01f * v.w;
  }
  __syncthreads();
  const int t = t0 + threadIdx.x;
  if (t >= y_len) return;
  float acc = 0.f;
  if (t < lim) {
#pragma unroll
    for (int k = 0; k < 7; ++k)
#pragma unroll 8
      for (int ci = 0; ci < C; ++ci) acc = fmaf(ws[k][ci], xs[ci][threadIdx.x + k], acc);
    acc = tanhf(acc);
  }
  y[(size_t)b * y_bs + t] = acc;
}

// [B][C][pitch] <-> [B][pitch][C] tiled transpose (32x32 through shared memory); T = __half reads an fp16 source
// (the generator's debug taps in precision mode 3) and writes fp32
template <class T = float>
__global__ void __launch_bounds__(256) transpose_kernel(const T* __restrict__ src, float* __restrict__ dst, int rows,
                                                        int cols, long long bs) {
  __shared__ float tile[32][33];
  const T* s = src + (size_t)blockIdx.z * bs;
  float* d = dst + (size_t)blockIdx.z * bs;
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int i = ty; i < 32; i += 8) {
    const int r = r0 + i, c = c0 + tx;
    tile[i][tx] = (r < rows && c < cols) ? static_cast<float>(s[(size_t)r * cols + c]) : 0.f;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, r = r0 + tx;
    if (r < rows && c < cols) d[(size_t)c * rows + r] = tile[tx][i];
  }
}

}  // namespace ovc
