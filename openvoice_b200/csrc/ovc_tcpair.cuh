// ovc_tcpair.cuh -- one ResBlock conv PAIR of the narrow generator stages (C = 64 / 32) in one persistent kernel:
//
//   t = c1(lrelu(x))  (k taps, dilation d)        modules.py:296-309, models.py:280-286
//   y = (c2(lrelu(t)) + x [+ y_old]) * scale      (k taps, dilation 1; residual, MRF accumulate and average fused)
//
// The intermediate t never leaves the SM: the epilogue of conv 1 (TMEM -> registers -> bias, leaky-relu, fp16 hi/lo
// split) writes it straight into the shared-memory A operand of conv 2.  HBM traffic of a pair drops from
// (x, t) + (t, x, y) = 5 passes to (x, x-as-residual [L2-hot], y) -- these layers are HBM-bound at k = 3 and close to
// it at k = 7 (DESIGN.md section 4.1).  Same arithmetic as two tcconv_kernel launches (3xFP16 split precision, stacked
// B operand, low-order accumulator), same operand layouts, same weight packing.
//
// Measured on a B200 (32 x 10 s, C = 32 stage, per pair): k = 3 0.84 ms fused vs 0.53 + 0.59 ms as two launches; k = 7
// 1.24 vs 1.27; k = 11 1.74 vs 1.64 -- the k >= 7 layers are bound by shared-memory operand reads, not by HBM, and pay
// for the 118 / 128 tile efficiency.  The host therefore fuses the k <= 5 pairs only (launch_pair / pair_fits): at C = 32,
// and at C = 64 for k = 3, whose weights (2 x 48 KB) stay resident next to the operand tiles with a halo of at most 8
// steps and ONE A2 buffer (TcpCfg<64>).  Larger C = 64 pairs do not fit, and with streamed weights a 118-step tile
// re-streams twice the weight bytes per step (measured 2x slower).
//
// Tile = 128 conv-1 steps; conv 2 needs H2 = (k-1)/2 steps of t on either side, so a tile yields R = 128 - 2*H2 output
// steps (k = 11: 118, 8 % of the MMA rows recomputed by the neighbours) and conv 1 reads 128 + 2*H1 steps of x.
// Warp roles (512 threads, one CTA per SM):
//   warp 0      weights of BOTH convs by TMA bulk copies, resident in shared memory for the whole launch (C = 32: 2 x 22
//               slots of 2 KB at k = 11; the host uses this kernel only when they fit)
//   warp 15     x chunks (rows x 32 channels) by tensor-map TMA into raw fp32 stages
//   warps 3-6   converters: raw -> lrelu -> hi/lo -> A1 operand (rows outside the utterance = 0)
//   warps 1, 2  MMA issuers of conv 1 / conv 2: conv 1 of the next tile runs on the tensor pipe while the epilogue of
//               conv 1 of this tile builds the A2 operand (two accumulator sets each)
//   warps 7-10  E1: accumulator of conv 1 -> A2 operand
//   warps 11-14 E2: accumulator of conv 2 -> bias, residual, accumulate, scale -> global (tc_epilogue)
#pragma once
#include "ovc_tcconv.cuh"

namespace ovc {

struct TcPairArgs {
  const float* x; long long x_bs;          // [B][Lpitch][C] fp32 channels-last: conv-1 input AND the residual
  const uint16_t* w1; const uint16_t* w2;  // packed weight slots of the two convs (pack_tc layout with TN = C)
  const float* bias1; const float* bias2;
  float* y; long long y_bs;                // [B][Lpitch][C]
  const long long* lens; int tmax; int mul;   // valid steps = min(tmax, lens[b]) * mul
  int C; int K; int DIL1;
  float slope;                             // leaky_relu slope of both convs' inputs
  float scale; int accumulate;
  int passes;
};

template <int TN>
struct TcpCfg {
  static_assert(TN == 32 || TN == 64, "C = 32 (k <= 11, halo <= 25) or C = 64 (k = 3, halo <= 8)");
  static constexpr int KCH = 32;
  // both convs' weights stay resident: C = 32: 2 x 22 slots of 2 KB (k <= 11); C = 64: 2 x 12 slots of 4 KB (k = 3 only),
  // which leaves room for operand tiles with a halo of at most 8 steps and ONE A2 buffer
  static constexpr int HMAX = TN == 32 ? 25 : 8;                  // (k - 1) / 2 * dilation of conv 1
  static constexpr int RAW_ROWS = TN == 32 ? 184 : 144;           // 128 + 2 * HMAX rounded up to 8
  static constexpr int ROWS1 = RAW_ROWS + 10, ROWS2 = 146;        // operand pitches in rows, = 2 (mod 8)
  static constexpr int NA1 = 2;
  static constexpr int NA2 = TN == 32 ? 2 : 1;
  static constexpr int NRAW = 2;
  static constexpr int RING = TN == 32 ? 44 : 24;                 // resident weight slots: 2 convs x (C / 16) x k
  static constexpr int SLOT_BYTES = 2 * 2 * TN * 16;
  static constexpr int A1_BYTES = 2 * 4 * ROWS1 * 16;
  static constexpr int A2_BYTES = 2 * (TN / 8) * ROWS2 * 16;
  static constexpr int RAW_STAGE_BYTES = RAW_ROWS * 128;          // multiple of 1024: every stage keeps the swizzle phase
  static_assert(RAW_STAGE_BYTES % 1024 == 0 && ROWS1 % 8 == 2, "stage / pitch alignment");
  static constexpr int NBARS = 2 * NA1 + 2 * NA2 + 2 * RING + 8 + 2 * NRAW;
  static constexpr size_t SMEM_BYTES = 1024 + NA1 * A1_BYTES + NA2 * A2_BYTES + RING * SLOT_BYTES + 1024 + NRAW * RAW_STAGE_BYTES;
  static constexpr uint32_t TMEM_COLS = 8 * TN;                   // 2 sets x (main + low) x TN for each conv
};

template <int TN>
__global__ void __launch_bounds__(TCN_THREADS, 1) tcpair_kernel(const TcPairArgs a, int n_tt, int total,
                                                                const __grid_constant__ CUtensorMap tmap) {
  using Cfg = TcpCfg<TN>;
  constexpr int ROWS1 = Cfg::ROWS1, ROWS2 = Cfg::ROWS2, NA1 = Cfg::NA1, NA2 = Cfg::NA2, NRAW = Cfg::NRAW, RING = Cfg::RING;
  constexpr int NKC2 = TN / 8;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
  uint64_t* a1_full = bars, *a1_empty = a1_full + NA1, *a2_full = a1_empty + NA1, *a2_empty = a2_full + NA2,
            *b_full = a2_empty + NA2, *b_empty = b_full + RING, *acc1_full = b_empty + RING, *acc1_empty = acc1_full + 2,
            *acc2_full = acc1_empty + 2, *acc2_empty = acc2_full + 2, *raw_full = acc2_empty + 2, *raw_empty = raw_full + NRAW;
  static_assert(Cfg::NBARS * 8 + 8 <= 1024, "barrier area");
  static_assert(Cfg::SMEM_BYTES <= 232448, "shared memory budget");
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(raw_empty + NRAW);
  unsigned char* a1buf = smem_raw + 1024;
  unsigned char* a2buf = a1buf + NA1 * Cfg::A1_BYTES;
  unsigned char* bring = a2buf + NA2 * Cfg::A2_BYTES;
  unsigned char* raw = bring + RING * Cfg::SLOT_BYTES;
  raw += (1024u - (smem_u32(raw) & 1023u)) & 1023u;

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int H1 = (a.K - 1) / 2 * a.DIL1, H2 = (a.K - 1) / 2;
  const int R = 128 - 2 * H2;                       // output steps per tile
  const int rows8 = (128 + 2 * H1 + 7) & ~7;        // staged rows of x per chunk
  const int nq = a.C / Cfg::KCH;
  const int n_slots = (a.C / 16) * a.K;             // weight slots per conv
  if (2 * n_slots > RING || H1 > Cfg::HMAX) __trap();   // weights resident, halo inside the staged rows (host: pair_fits)
  const bool three = a.passes == 3;

  if (tid == 0) {
    for (int i = 0; i < NA1; ++i) { mbar_init(&a1_full[i], 128); mbar_init(&a1_empty[i], 1); }
    for (int i = 0; i < NA2; ++i) { mbar_init(&a2_full[i], 128); mbar_init(&a2_empty[i], 1); }
    for (int i = 0; i < RING; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc1_full[i], 1); mbar_init(&acc1_empty[i], 4);
      mbar_init(&acc2_full[i], 1); mbar_init(&acc2_empty[i], 4);
    }
    for (int i = 0; i < NRAW; ++i) { mbar_init(&raw_full[i], 1); mbar_init(&raw_empty[i], 128); }
    fence_mbar_init();
  }
  // rows of the A2 operand that conv 1 never produces (the taps of the discarded last output rows read them): zero once
  for (int i = tid; i < NA2 * Cfg::A2_BYTES / 16; i += TCN_THREADS)
    reinterpret_cast<uint4*>(a2buf)[i] = make_uint4(0u, 0u, 0u, 0u);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  if (warp == 1) tc::tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  tc::fence_before();
  __syncthreads();
  tc::fence_after();
  const uint32_t tmem_d = *tmem_slot;
  const uint32_t acc1_base = tmem_d, acc2_base = tmem_d + 4 * TN;

  // every role walks the same tile sequence: tiles of R output steps (tc_tile)
  if (warp == 0) {
    // ------------------------------------------------------------ weights of both convs
    if (lane == 0) {
      tc_load_resident<Cfg::SLOT_BYTES>(bring, b_full, a.w1, n_slots);
      tc_load_resident<Cfg::SLOT_BYTES>(bring + n_slots * Cfg::SLOT_BYTES, b_full + n_slots, a.w2, n_slots);
    }
  } else if (warp == 15) {
    // ------------------------------------------------------------ x chunks by tensor-map TMA
    if (lane == 0) {
      int st = 0;
      uint32_t phase = 1;
      const uint32_t box_bytes = (uint32_t)rows8 * 128u;
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const TcTile tl = tc_tile(tile, n_tt, R, a.lens, nullptr, a.tmax, a.mul);
        if (tl.t0 >= tl.lim) continue;
        for (int q = 0; q < nq; ++q) {
          mbar_wait(&raw_empty[st], phase);
          mbar_expect_tx(&raw_full[st], box_bytes);
          tma_tensor3d_g2s(raw + st * Cfg::RAW_STAGE_BYTES, &tmap, q * Cfg::KCH, tl.t0 - H2 - H1, tl.b, &raw_full[st]);
          if (++st == NRAW) { st = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1 || warp == 2) {
    // ------------------------------------------------------------ MMA issuers (converged warps, elected lane issues):
    // warp 1 issues conv 1, warp 2 conv 2 -- one thread cannot feed the tensor pipe at N <= 64 (an MMA pair lasts 88
    // cycles).  Conv 1 of tile i+1 runs on the tensor pipe while E1 builds the A2 operand of tile i.
    constexpr uint32_t LBO1 = ROWS1 * 16, LBO2 = ROWS2 * 16, LBO_B = 2 * TN * 16, SBO = 128;
    constexpr uint32_t A1_LO16 = (4 * ROWS1 * 16) >> 4, A2_LO16 = (NKC2 * ROWS2 * 16) >> 4, SLOT16 = Cfg::SLOT_BYTES >> 4;
    const uint64_t a1_proto = tc::make_desc(0, LBO1, SBO), a2_proto = tc::make_desc(0, LBO2, SBO), b_proto = tc::make_desc(0, LBO_B, SBO);
    const uint64_t b_ring = b_proto + (tc::smem_addr(bring) >> 4);
    const uint32_t dil = (uint32_t)a.DIL1;
    const int conv = warp - 1;
    for (int it = 0; it < n_slots; ++it) mbar_wait(&b_full[conv * n_slots + it], 0u);   // resident weights: waited on once
    tc::fence_after();
    if (warp == 1) {
      int buf1 = 0, n1 = 0;
      uint32_t a1phase = 0;
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const TcTile tl = tc_tile(tile, n_tt, R, a.lens, nullptr, a.tmax, a.mul);
        if (tl.t0 >= tl.lim) continue;
        const int set = n1 & 1;
        mbar_wait(&acc1_empty[set], ((n1 >> 1) & 1) ^ 1);
        tc::fence_after();
        const uint32_t acc = acc1_base + set * 2 * TN;
        bool first = true;
        for (int q = 0; q < nq; ++q) {
          mbar_wait(&a1_full[buf1], a1phase);
          tc::fence_after();
          for (int j = 0; j < 2; ++j) {
            uint64_t a_cur = a1_proto + ((tc::smem_addr(a1buf + buf1 * Cfg::A1_BYTES) + 2 * j * LBO1) >> 4);
            uint64_t b_slot = b_ring + (uint32_t)((q * 2 + j) * a.K) * SLOT16;
            for (int tap = 0; tap < a.K; ++tap) {
              if (tc::elect_one()) tc_mma_step<TN>(acc, a_cur, A1_LO16, b_slot, three, !first);
              __syncwarp();
              first = false;
              a_cur += dil;
              b_slot += SLOT16;
            }
          }
          if (tc::elect_one()) tc::mma_commit(&a1_empty[buf1]);
          __syncwarp();
          if (++buf1 == NA1) { buf1 = 0; a1phase ^= 1; }
        }
        if (tc::elect_one()) tc::mma_commit(&acc1_full[set]);
        __syncwarp();
        ++n1;
      }
    } else {
      int n2 = 0;
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const TcTile tl = tc_tile(tile, n_tt, R, a.lens, nullptr, a.tmax, a.mul);
        if (tl.t0 >= tl.lim) continue;
        const int set = n2 & 1, buf2 = n2 % NA2;
        mbar_wait(&acc2_empty[set], ((n2 >> 1) & 1) ^ 1);
        mbar_wait(&a2_full[buf2], (n2 / NA2) & 1);
        tc::fence_after();
        const uint32_t acc = acc2_base + set * 2 * TN;
        bool first = true;
        uint64_t b_slot = b_ring + (uint32_t)n_slots * SLOT16;
        for (int kk = 0; kk < a.C / 16; ++kk) {
          uint64_t a_cur = a2_proto + ((tc::smem_addr(a2buf + buf2 * Cfg::A2_BYTES) + 2 * kk * LBO2) >> 4);
          for (int tap = 0; tap < a.K; ++tap) {
            if (tc::elect_one()) tc_mma_step<TN>(acc, a_cur, A2_LO16, b_slot, three, !first);
            __syncwarp();
            first = false;
            a_cur += 1;             // conv 2 has dilation 1
            b_slot += SLOT16;
          }
        }
        if (tc::elect_one()) {
          tc::mma_commit(&a2_empty[buf2]);
          tc::mma_commit(&acc2_full[set]);
        }
        __syncwarp();
        ++n2;
      }
    }
  } else if (warp >= 3 && warp <= 6) {
    // ------------------------------------------------------------ converters: x -> A1 operand
    const int pt = tid - 96;
    const int items = rows8 * 4;
    int buf = 0, st = 0;
    uint32_t ephase = 1, rphase = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
      const TcTile tl = tc_tile(tile, n_tt, R, a.lens, nullptr, a.tmax, a.mul);
      if (tl.t0 >= tl.lim) continue;
      for (int q = 0; q < nq; ++q) {
        mbar_wait(&raw_full[st], rphase);
        mbar_wait(&a1_empty[buf], ephase);
        tc_convert_raw<ROWS1, 128>(raw + st * Cfg::RAW_STAGE_BYTES, a1buf + buf * Cfg::A1_BYTES, pt, items, tl.t0 - H2 - H1, tl.lim,
                                   a.slope);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_arrive(&a1_full[buf]);
        if (++buf == NA1) { buf = 0; ephase ^= 1; }
        mbar_arrive(&raw_empty[st]);
        if (++st == NRAW) { st = 0; rphase ^= 1; }
      }
    }
  } else if (warp >= 7 && warp <= 10) {
    // ------------------------------------------------------------ E1: accumulator of conv 1 -> A2 operand of conv 2
    const int lane_base = (warp & 3) * 32;
    const int rsub = lane >> 2, csub = (lane & 3) * 2;
    int n = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
      const TcTile tl = tc_tile(tile, n_tt, R, a.lens, nullptr, a.tmax, a.mul);
      if (tl.t0 >= tl.lim) continue;
      const int set = n & 1, buf2 = n % NA2;
      mbar_wait(&a2_empty[buf2], ((n / NA2) & 1) ^ 1);     // conv 2 of the tile that used this A2 buffer has read it
      mbar_wait(&acc1_full[set], (n >> 1) & 1);
      tc::fence_after();
      unsigned char* a2h = a2buf + buf2 * Cfg::A2_BYTES;
      unsigned char* a2l = a2h + NKC2 * ROWS2 * 16;
      const uint32_t acc = acc1_base + set * 2 * TN;
#pragma unroll 1
      for (int c0 = 0; c0 < TN; c0 += 32) {
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
          const int row_a = lane_base + 16 * h + rsub, row_b = row_a + 8;     // conv-1 output rows = A2 rows
          const uint32_t taddr = acc + ((uint32_t)(lane_base + 16 * h) << 16) + c0;
          uint32_t rm[16], rl[16];
          tc::tmem_ld16x256_x4_issue(taddr, rm);
          if (three) tc::tmem_ld16x256_x4_issue(taddr + TN, rl);
          float2 bq[4];
#pragma unroll
          for (int g = 0; g < 4; ++g) bq[g] = __ldg(reinterpret_cast<const float2*>(a.bias1 + c0 + 8 * g + csub));
          float v[16];
          if (three) {
            tc::tmem_ld_wait16x2(rm, rl);
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = fmaf(__uint_as_float(rl[i]), tc::kLoInv, __uint_as_float(rm[i]));
          } else {
            tc::tmem_ld_wait16(rm);
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(rm[i]);
          }
          // t lives on steps [0, lim): outside them conv 2 sees zero padding, not conv 1 evaluated on padding
          const int ta = tl.t0 - H2 + row_a, tb = ta + 8;
          const bool oka = ta >= 0 && ta < tl.lim, okb = tb >= 0 && tb < tl.lim;
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            float x0 = v[4 * g] + bq[g].x, x1 = v[4 * g + 1] + bq[g].y, x2 = v[4 * g + 2] + bq[g].x, x3 = v[4 * g + 3] + bq[g].y;
            x0 = oka ? fmaxf(x0, x0 * a.slope) : 0.f;
            x1 = oka ? fmaxf(x1, x1 * a.slope) : 0.f;
            x2 = okb ? fmaxf(x2, x2 * a.slope) : 0.f;
            x3 = okb ? fmaxf(x3, x3 * a.slope) : 0.f;
            __half2 ha, la, hb, lb;
            tc::split_f16x2(x0, x1, ha, la);
            tc::split_f16x2(x2, x3, hb, lb);
            const int kc = (c0 >> 3) + g;
            const int oa = (kc * ROWS2 + row_a) * 16 + (lane & 3) * 4, ob = (kc * ROWS2 + row_b) * 16 + (lane & 3) * 4;
            *reinterpret_cast<__half2*>(a2h + oa) = ha;
            *reinterpret_cast<__half2*>(a2h + ob) = hb;
            *reinterpret_cast<__half2*>(a2l + oa) = la;
            *reinterpret_cast<__half2*>(a2l + ob) = lb;
          }
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes -> tensor-core (async) proxy
      mbar_arrive(&a2_full[buf2]);
      tc::fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc1_empty[set]);
      ++n;
    }
  } else if (warp >= 11 && warp <= 14) {
    // ------------------------------------------------------------ E2: accumulator of conv 2 -> global
    TcConvArgs e{};
    e.y = a.y; e.y_bs = a.y_bs; e.y_ld = TN;
    e.r = a.x;                       // the pair's input is its residual (same geometry as y)
    e.bias = a.bias2; e.bias_bs = 0;
    e.epi = 0; e.accumulate = a.accumulate; e.scale = a.scale; e.passes = a.passes;
    int n = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
      const TcTile tl = tc_tile(tile, n_tt, R, a.lens, nullptr, a.tmax, a.mul);
      if (tl.t0 >= tl.lim) continue;
      const int set = n & 1;
      tc_epilogue<TN>(e, acc2_base + set * 2 * TN, tl.b, tl.t0, 0, min(tl.lim, tl.t0 + R), warp, lane, 0, 1, 0, TN, &acc2_full[set],
                      (n >> 1) & 1);
      tc::fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc2_empty[set]);
      ++n;
    }
  }
  tc::fence_before();
  __syncthreads();
  if (warp == 1) tc::tmem_dealloc(tmem_d, Cfg::TMEM_COLS);
}

}  // namespace ovc
