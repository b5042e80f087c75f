// dahitra_b200 — pixel decoder on the tensor cores (tcgen05, TF32 operands, fp32 accumulate in TMEM).
//
// Same algebra as decoder.cu (collapsed cross-attention + MLP, reference models/help_funcs.py:66-114,170-186),
// re-mapped so that the four 128x32x32 products of every layer run as tcgen05.mma and everything that is
// per-pixel (LayerNorm statistics, the 4-key softmax per head, exact-erf GELU) is thread-local:
//   * a warpgroup owns 128 pixels; thread t owns pixel t = TMEM lane t, so `tcgen05.ld.32x32b` hands each thread the
//     32 channels of ITS pixel — no shuffles anywhere.
//   * the running activation x lives in TMEM columns [0,32) for the whole call; attention and MLP outputs are
//     accumulated INTO it by the MMA (x += P.Bv, x += G.W2).  Biases are pixel-independent, so they are applied
//     as host-precomputed cumulative vectors when x is read back (no TMEM write-back).
//   * A operands (xhat, P, xhat', G) never touch shared memory: each thread writes its row with ONE
//     `tcgen05.st.32x32b.x32` into TMEM columns [32,64) (TF32 hi) / [64,96) (lo) and the MMA reads A from tensor
//     memory (`tcgen05.mma [d], [a], bdesc`).  No swizzled stores, no proxy fence, and the MMA's shared-memory
//     traffic is only the 1 KB B slice per K step.  B operands (per-image tables, shared MLP weights) arrive
//     pre-swizzled from global memory through 1-D bulk copies (double-buffered, prefetched one layer ahead).
//   * X3 = true: error-compensated "3xTF32".  Every operand is split v = hi + lo with hi exactly representable
//     in TF32 (A: cvt.rna on the fly, written to the second column block; B: split by the table kernel / on the
//     host) and each product is issued as A_hi.B_hi + A_lo.B_hi + A_hi.B_lo — fp32-grade accuracy.
// Per layer: 4 x {tcgen05.st A row, barrier, one thread issues the MMAs + commit, mbarrier wait, tcgen05.ld}.
// A CTA holds four warpgroups (4 x 128 TMEM columns = the whole tensor memory) whose serial chains overlap.
#include "tc_common.cuh"
#include <type_traits>

using namespace dhtc;

namespace {

__device__ __forceinline__ float tf32_hi(float v) { return tf32_round(v); }

__device__ __forceinline__ float ex2_approx(float x) {      // MUFU.EX2, relative error <= 2^-22
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {      // MUFU.RCP, <= 1 ulp
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// GELU(h) = h * Phi(h) with the exact-erf Phi of the reference (nn.GELU default, help_funcs.py:36-47), evaluated
// branch-free:  Phi(-u) = 2^g(u), g = degree-8 weighted-minimax fit of log2(erfc(u / sqrt 2) / 2) on [0, 6]
// (tools/fit_gelu.py), Phi(h) = h >= 0 ? 1 - Phi(-|h|) : Phi(-|h|).  Measured against the fp64 GELU over [-8, 8]:
// max abs error 3.8e-7 (4.5e-8 for |h| <= 0.5) — the same as the fp32 formula 0.5 h (1 + erff(h / sqrt 2)), at a third
// of its instruction count (erff is two divergent polynomial branches + an exp).
__device__ __forceinline__ float gelu_phi8(float h) {
  const float u = fminf(fabsf(h), 6.0f);
  float g = -1.966050149e-06f;
  g = fmaf(g, u, 2.892093107e-05f);
  g = fmaf(g, u, -1.361643517e-04f);
  g = fmaf(g, u, -2.589166979e-04f);
  g = fmaf(g, u, 7.225090638e-03f);
  g = fmaf(g, u, -5.261069164e-02f);
  g = fmaf(g, u, -4.591687918e-01f);
  g = fmaf(g, u, -1.151110411e+00f);
  g = fmaf(g, u, -9.999998808e-01f);
  const float q = ex2_approx(g);
  return h * (h >= 0.f ? 1.0f - q : q);
}

// the same on a pair of values: the Horner chain and the final products are packed FFMA2 / FMUL2 (one issued instruction per
// two values; this kernel is bound by instruction issue), |h|, 2^g and the sign select stay scalar
__device__ __forceinline__ float2 gelu_phi8_2(float2 h) {
  const float2 u = make_float2(fminf(fabsf(h.x), 6.0f), fminf(fabsf(h.y), 6.0f));
  float2 g = f2_bcast(-1.966050149e-06f);
  g = ffma2(g, u, f2_bcast(2.892093107e-05f));
  g = ffma2(g, u, f2_bcast(-1.361643517e-04f));
  g = ffma2(g, u, f2_bcast(-2.589166979e-04f));
  g = ffma2(g, u, f2_bcast(7.225090638e-03f));
  g = ffma2(g, u, f2_bcast(-5.261069164e-02f));
  g = ffma2(g, u, f2_bcast(-4.591687918e-01f));
  g = ffma2(g, u, f2_bcast(-1.151110411e+00f));
  g = ffma2(g, u, f2_bcast(-9.999998808e-01f));
  const float qx = ex2_approx(g.x), qy = ex2_approx(g.y);
  return fmul2(h, make_float2(h.x >= 0.f ? 1.0f - qx : qx, h.y >= 0.f ? 1.0f - qy : qy));
}

// ----------------------------------------------------------------------------------------------------
// table builder (TC layout): per (image-call, layer)  DH_TABTC_FLOATS =
//     [TA_hi swz 32x32][TB_hi swz 32x32][cA 32] [TA_lo swz][TB_lo swz]
//   TA[n = h*4+j][k = c] = g_c * sum_c' Mqk[h][c][c'] mn_j[c']       (B operand of  S = xhat . TA^T)
//   TB[n = c][k = h*4+j] =       sum_c' Mov[h][c][c'] mn_j[c']       (B operand of  x += P . TB^T)
//   cA[h*4+j]            = sum_c b_c * (TA/g)[h*4+j][c]
//   TA and cA carry a factor log2(e): the decoder's softmax is 2^(s - max) on MUFU.EX2 with no per-element scaling.
//   hi = TF32-rounded value, lo = TF32-rounded remainder (used by the 3xTF32 decoder only)
// ----------------------------------------------------------------------------------------------------
__device__ __forceinline__ float ln_lane32(float v, float g, float b) {
  const float mu = warp_sum(v) * (1.f / 32.f);
  const float d = v - mu;
  const float var = warp_sum(d * d) * (1.f / 32.f);
  return d * (1.0f / sqrtf(var + 1e-5f)) * g + b;
}

__global__ void __launch_bounds__(128)
decoder_tables_tc_kernel(const float* __restrict__ mem, int B, int first_call, const float* __restrict__ dec, int heads,
                         float* __restrict__ tables, int depth) {
  __shared__ float MN[4][32];
  extern __shared__ __align__(16) float dt_w[];               // Mqk | Mov of this layer: 2 * heads * 1024 floats
  const int lane = threadIdx.x & 31, j = threadIdx.x >> 5;
  const int layer = blockIdx.x;
  const int ci = blockIdx.y / B, pair = blockIdx.y % B;
  const int call = first_call + ci;
  const float* L = dec + (size_t)layer * DH_DEC_LAYER_FLOATS(heads);
  // the layer's matrices are cold in L2 (see token_encoder_kernel): one asynchronous fetch instead of 4 * heads
  // dependent batches of loads
  {
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(dt_w);
    for (int i = threadIdx.x; i < heads * 512; i += 128)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + (uint32_t)i * 16u), "l"(L + 64 + (size_t)i * 4) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  const float* MqkT = dt_w;
  const float* MovT = MqkT + (size_t)heads * 1024;
  float* T = tables + ((size_t)blockIdx.y * depth + layer) * DH_TABTC_FLOATS;
  float* TA = T; float* TB = T + 1024; float* cA = T + 2048; float* TAl = T + 2080; float* TBl = T + 2080 + 1024;
  const float g = __ldg(L + lane), b = __ldg(L + 32 + lane);
  dh_pdl_wait();                       // `mem` comes from the token encoder launched just before
  dh_pdl_launch_dependents();
  MN[j][lane] = ln_lane32(__ldg(mem + ((size_t)pair * 3 + call) * 128 + j * 32 + lane), g, b);
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  for (int h = 0; h < heads; ++h) {
    const float* mq = MqkT + (size_t)h * 1024;
    const float* mv = MovT + (size_t)h * 1024;
    float a = 0.f, v = 0.f;
#pragma unroll 8
    for (int c2 = 0; c2 < 32; ++c2) {
      const float mn = MN[j][c2];
      a = fmaf(mq[c2 * 32 + lane], mn, a);
      v = fmaf(mv[c2 * 32 + lane], mn, v);
    }
    const int hj = h * 4 + j;
    a *= 1.4426950408889634f;                               // log2(e)
    const float ga = g * a;
    const float ga_hi = tf32_hi(ga), v_hi = tf32_hi(v);
    TA[sw128_idx(hj, lane)] = ga_hi;
    TAl[sw128_idx(hj, lane)] = tf32_hi(ga - ga_hi);
    TB[sw128_idx(lane, hj)] = v_hi;
    TBl[sw128_idx(lane, hj)] = tf32_hi(v - v_hi);
    const float ca = warp_sum(b * a);
    if (lane == 0) cA[hj] = ca;
  }
  if (heads == 4 && j == 0 && lane >= 16) cA[lane] = 0.f;
}

// ----------------------------------------------------------------------------------------------------
// decoder
// ----------------------------------------------------------------------------------------------------
constexpr int PDT_ROWS = 128;
constexpr uint32_t PDT_TAB_HI = 2080 * 4;                   // TA_hi | TB_hi | cA
constexpr uint32_t PDT_MLP_HI = 2144 * 4;                   // W1_hi | W2_hi | b1f | cbA | cbM
constexpr uint32_t PDT_LO = 2048 * 4;                       // two 32x32 lo tiles
constexpr uint32_t PDT_HI_STRIDE = 9216;                    // 1024-aligned room for a hi block
constexpr int PDT_G = 4;                                    // warpgroups (tiles) per CTA
#ifndef PDT_A_ROUND
#define PDT_A_ROUND 1          // 0: truncation split (3 % faster decoder, 2^-21 instead of 2^-22 per operand: measured 5.7e-4 vs 5.5e-4 whole-net)
#endif
#ifndef PDT_TURN_D
#define PDT_TURN_D 2
#endif
constexpr uint32_t PDT_WG_COLS = 128;                       // TMEM columns per warpgroup: x | A_hi | A_lo | D
constexpr uint32_t TM_X = 0, TM_A = 32, TM_AL = 64, TM_D = 96;

// A CTA holds G warpgroups; each owns one 128-pixel tile (128 TMEM columns, its own MMA barrier) of the SAME image,
// so all of them share the per-layer table / MLP buffers.  G independent serial chains per CTA are what hides the
// st-A -> MMA -> tcgen05.ld latency of each chain.
template <bool X3> struct PdtCfg {
  static constexpr int G = PDT_G;
  static constexpr uint32_t BUF = PDT_HI_STRIDE + (X3 ? PDT_LO : 0);            // one table (or MLP) buffer
  static constexpr int NB = 3;                                                  // table / MLP buffers (layers in flight)
  static constexpr uint32_t OFF_IO = 2 * NB * BUF;                 // per-warp 32 x 128 B transpose buffers for the global I/O
  static constexpr uint32_t SMEM = OFF_IO + PDT_G * 4 * 4096 + 1024;
};

template <int HEADS, bool X3>
__global__ void __launch_bounds__(PDT_ROWS * PdtCfg<X3>::G, 1)
pixel_decoder_tc_kernel(const float* __restrict__ x, const float* __restrict__ pos, const float* __restrict__ tables,
                        const float* __restrict__ pack, int npix, int w, int depth, const float* __restrict__ skip,
                        int skip_up, float* __restrict__ out, long long out_split_plane, int h16) {
  using Cfg = PdtCfg<X3>;
  constexpr int H4 = HEADS * 4;
  constexpr uint32_t IDESC_S = umma_idesc_tf32(128, H4);
  constexpr uint32_t IDESC_32 = umma_idesc_tf32(128, 32);
  extern __shared__ uint8_t pdt_raw[];
  constexpr int G = Cfg::G;
  constexpr int NB = Cfg::NB;
  __shared__ __align__(8) uint64_t tab_bar[NB], free_bar[NB], mma_bar[G];
  __shared__ uint32_t tmem_slot;

  const int wg = threadIdx.x >> 7;                                      // warpgroup = tile within the CTA
  const int tid = threadIdx.x & 127, warp = tid >> 5, img = blockIdx.y; // tid: row of this warpgroup's tile
  const uint32_t base = (smem_u32(pdt_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = pdt_raw + (base - smem_u32(pdt_raw));
  constexpr uint32_t BUFS0 = 0;
  auto tab_addr = [&](int b) { return base + BUFS0 + (uint32_t)b * Cfg::BUF; };
  auto mlp_addr = [&](int b) { return base + BUFS0 + NB * Cfg::BUF + (uint32_t)b * Cfg::BUF; };
  auto tab_ptr = [&](int b) { return reinterpret_cast<const float*>(base_ptr + BUFS0 + (size_t)b * Cfg::BUF); };
  auto mlp_ptr = [&](int b) { return reinterpret_cast<const float*>(base_ptr + BUFS0 + NB * Cfg::BUF + (size_t)b * Cfg::BUF); };

  if (threadIdx.x == 0) {
    for (int i = 0; i < NB; ++i) { mbar_init(smem_u32(&tab_bar[i]), 1); mbar_init(smem_u32(&free_bar[i]), G); }
    for (int i = 0; i < G; ++i) mbar_init(smem_u32(&mma_bar[i]), 1);
    mbar_fence_init();
  }
  if (threadIdx.x < 32) tmem_alloc(smem_u32(&tmem_slot), 512);          // G x 128 columns
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  dh_pdl_wait();                       // tables / x / skip come from earlier launches of the stream
  dh_pdl_launch_dependents();
  const uint32_t tmem_wg = tmem_slot + (uint32_t)wg * PDT_WG_COLS;      // this warpgroup's columns
  const uint32_t tmem = tmem_wg + ((uint32_t)(warp * 32) << 16);       // ... and this warp's lane quarter
  const uint32_t my_bar = smem_u32(&mma_bar[wg]);

  auto issue_loads = [&](int layer) {
    const int b = layer % NB;
    const uint32_t bar = smem_u32(&tab_bar[b]);
    const float* tg = tables + ((size_t)img * depth + layer) * DH_TABTC_FLOATS;
    const float* pg = pack + (size_t)layer * DH_DECTC_LAYER_FLOATS;
    mbar_expect_tx(bar, PDT_TAB_HI + PDT_MLP_HI + (X3 ? 2 * PDT_LO : 0));
    bulk_load_1d(tab_addr(b), tg, PDT_TAB_HI, bar);
    bulk_load_1d(mlp_addr(b), pg, PDT_MLP_HI, bar);
    if (X3) {
      bulk_load_1d(tab_addr(b) + PDT_HI_STRIDE, tg + 2080, PDT_LO, bar);
      bulk_load_1d(mlp_addr(b) + PDT_HI_STRIDE, pg + 2144, PDT_LO, bar);
    }
  };
  if (threadIdx.x == 0) {
    issue_loads(0);
    if (depth > 1) issue_loads(1);
  }
  // the MMA-issuing thread of warpgroup g sits in its warp g, so the four issuers run on four different schedulers
  const bool issuer = (tid == 32 * wg);
  // ALU turn-taking (named barriers 5..8, 128 arriving + 128 waiting threads): identical warpgroups otherwise run in
  // lockstep — all in their ALU phase, then all waiting on the tensor pipe, then all on the TMEM read port — and the
  // phases add up instead of overlapping.  Warpgroup g may enter an ALU phase only after warpgroup g-TURN_D has left
  // its own; the rest of its chain (tcgen05.st drain, MMAs, commit, tcgen05.ld) runs while others hold the ALUs.
  constexpr int TURN_D = PDT_TURN_D;
  auto turn_wait = [&]() { if (TURN_D) asm volatile("bar.sync %0, 256;" ::"r"(5 + wg) : "memory"); };
  auto turn_pass = [&]() { if (TURN_D) asm volatile("bar.arrive %0, 256;" ::"r"(5 + ((wg + TURN_D) & 3)) : "memory"); };
  if (TURN_D && wg >= G - TURN_D) turn_pass();                         // the first TURN_D warpgroups start immediately

  // ---- x (+ pos) -> registers and TMEM.  Global I/O goes through a per-warp shared-memory transpose: 8 lanes read one
  // pixel's 128-byte row (4 whole lines per instruction), then every thread picks up ITS row — a thread-per-row access
  // would touch 32 different lines with every instruction.
  float* io = reinterpret_cast<float*>(base_ptr + Cfg::OFF_IO + (size_t)(threadIdx.x >> 5) * 4096);
  const int lane = threadIdx.x & 31, c8 = lane & 7, r8 = lane >> 3;
  const int pw0 = (blockIdx.x * G + wg) * PDT_ROWS + warp * 32;         // first pixel of this warp
  float2 xr[16];                                                        // this thread's pixel: 32 channels as 16 packed pairs
#pragma unroll
  for (int g = 0; g < 8; ++g) {
    const int r = g * 4 + r8, pr = pw0 + r;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (pr < npix) {
      if (h16) {                                                        // x is one FP16 plane: 4 channels = 8 bytes
        const uint2 u = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const uint16_t*>(x) + ((size_t)img * npix + pr) * 32 + c8 * 4));
        v = make_float4(f16_lo(u.x), f16_hi(u.x), f16_lo(u.y), f16_hi(u.y));
      } else {
        v = ldg4(x + ((size_t)img * npix + pr) * 32 + c8 * 4);
      }
      if (pos) { const float4 q = ldg4(pos + (size_t)pr * 32 + c8 * 4); v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w; }
    }
    *reinterpret_cast<float4*>(io + r * 32 + ((c8 ^ (r & 7)) << 2)) = v;
  }
  __syncwarp();
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float4 v = *reinterpret_cast<const float4*>(io + lane * 32 + ((q ^ (lane & 7)) << 2));
    xr[q * 2] = make_float2(v.x, v.y); xr[q * 2 + 1] = make_float2(v.z, v.w);
  }
  __syncwarp();
  {
    uint32_t u[32];
#pragma unroll
    for (int c = 0; c < 16; ++c) { u[2 * c] = __float_as_uint(xr[c].x); u[2 * c + 1] = __float_as_uint(xr[c].y); }
    tmem_st32(tmem + TM_X, u);
  }

  // this thread's row of the A operand -> tensor memory: TF32-rounded values and, for X3, the remainders
  // A operand rows.  X3: hi = v rounded to the nearest TF32 value, lo = v - hi (the tensor core truncates lo to TF32: the pair
  // carries v to 2^-22).  PDT_A_ROUND = 0 is the cheaper truncation split: the tensor core ignores the low 13 mantissa bits of an
  // fp32 word anyway, so hi = v as it is and lo = v - trunc(v) — one AND + one subtract per element instead of add, AND, subtract.
  auto write_a_row = [&](const float2 (&v)[16]) {
    uint32_t hi[32];
#if PDT_A_ROUND
#pragma unroll
    for (int c = 0; c < 16; ++c) { hi[2 * c] = __float_as_uint(tf32_hi(v[c].x)); hi[2 * c + 1] = __float_as_uint(tf32_hi(v[c].y)); }
#else
#pragma unroll
    for (int c = 0; c < 16; ++c) { hi[2 * c] = __float_as_uint(v[c].x); hi[2 * c + 1] = __float_as_uint(v[c].y); }
#endif
    tmem_st32(tmem + TM_A, hi);
    if (X3) {
      uint32_t lo[32];
#pragma unroll
      for (int c = 0; c < 16; ++c) {
#if PDT_A_ROUND
        const float2 l = fsub2(v[c], make_float2(__uint_as_float(hi[2 * c]), __uint_as_float(hi[2 * c + 1])));
#else
        const float2 l = fsub2(v[c], make_float2(__uint_as_float(hi[2 * c] & 0xFFFFE000u), __uint_as_float(hi[2 * c + 1] & 0xFFFFE000u)));
#endif
        lo[2 * c] = __float_as_uint(l.x); lo[2 * c + 1] = __float_as_uint(l.y);
      }
      tmem_st32(tmem + TM_AL, lo);
    }
  };
  // LayerNorm statistics of this thread's pixel: t = x - mean (packed), returns 1 / sqrt(var + eps)
  auto center = [&](const float2 (&x)[16], float2 (&t)[16]) -> float {
    float2 s2 = x[0];
#pragma unroll
    for (int c = 1; c < 16; ++c) s2 = fadd2(s2, x[c]);
    const float mu = (s2.x + s2.y) * (1.f / 32.f);
    const float2 nmu = f2_bcast(-mu);
    float2 v2 = make_float2(0.f, 0.f);
#pragma unroll
    for (int c = 0; c < 16; ++c) { t[c] = fadd2(x[c], nmu); v2 = ffma2(t[c], t[c], v2); }
    return rsqrtf((v2.x + v2.y) * (1.f / 32.f) + 1e-5f);
  };

  uint32_t mma_phase = 0;
  // one MMA round: all rows of the A block(s) are in TMEM -> thread 0 issues `nk` K-steps -> everyone waits for the commit.
  auto mma_round = [&](uint32_t b_hi_addr, uint32_t b_lo_addr, uint32_t idesc, uint32_t tm_col, auto nk_c, bool accumulate) {
    constexpr int nk = decltype(nk_c)::value;
    tc_fence_before();
    asm volatile("bar.sync %0, 128;" ::"r"(wg + 1) : "memory");         // this warpgroup's rows are all written
    if (issuer) {
      tc_fence_after();
      const uint64_t bh = umma_desc_sw128(b_hi_addr);
      const uint32_t d = tmem_wg + tm_col, ah = tmem_wg + TM_A, al = tmem_wg + TM_AL;
#pragma unroll
      for (int k = 0; k < nk; ++k) umma_tf32_ts(d, ah + 8u * k, bh + (uint64_t)(2 * k), idesc, (accumulate || k) ? 1u : 0u);
      if (X3) {
        const uint64_t bl = umma_desc_sw128(b_lo_addr);
#pragma unroll
        for (int k = 0; k < nk; ++k) umma_tf32_ts(d, al + 8u * k, bh + (uint64_t)(2 * k), idesc, 1u);
#pragma unroll
        for (int k = 0; k < nk; ++k) umma_tf32_ts(d, ah + 8u * k, bl + (uint64_t)(2 * k), idesc, 1u);
      }
      umma_commit(my_bar);
    }
    mbar_wait(my_bar, mma_phase);
    mma_phase ^= 1u;
    tc_fence_after();
  };
  using K4 = std::integral_constant<int, 4>;
  using KP = std::integral_constant<int, H4 / 8>;

  for (int layer = 0; layer < depth; ++layer) {
    const int b = layer % NB;
    // prefetch layer+2 into the buffer layer-1 used, once EVERY warpgroup has released it (free_bar counts G arrivals);
    // the warpgroups are otherwise free to drift apart by up to two layers, which is what staggers their chains
    if (threadIdx.x == 0 && layer + 2 < depth) {
      if (layer >= 1) mbar_wait(smem_u32(&free_bar[(layer + 2) % NB]), (uint32_t)(((layer - 1) / NB) & 1));
      issue_loads(layer + 2);
    }
    mbar_wait(smem_u32(&tab_bar[b]), (uint32_t)((layer / NB) & 1));
    const float* tabp = tab_ptr(b);
    const float* mlpp = mlp_ptr(b);
    const float* cA = tabp + 2048;
    const float* b1f = mlpp + 2048; const float* cbA = mlpp + 2080; const float* cbM = mlpp + 2112;
    const uint32_t t_hi = tab_addr(b), t_lo = tab_addr(b) + PDT_HI_STRIDE;
    const uint32_t m_hi = mlp_addr(b), m_lo = mlp_addr(b) + PDT_HI_STRIDE;
    float2 t[16];
    float rstd;
    const float2* cA2 = reinterpret_cast<const float2*>(cA);
    const float2* b1f2 = reinterpret_cast<const float2*>(b1f);
    const float2* cbA2 = reinterpret_cast<const float2*>(cbA);
    const float2* cbM2 = reinterpret_cast<const float2*>(cbM);
    // ---- 1. S = xhat . TA^T            (rstd is applied to the MMA result: S = rstd * ((x - mu) . TA) + cA)
    {
      turn_wait();
      rstd = center(xr, t);
      write_a_row(t);
      turn_pass();
    }
    mma_round(t_hi, t_lo, IDESC_S, TM_D, K4{}, false);
    // ---- 2. P = softmax_j(S + cA) ; x += P . TB^T
    {
      const float2 rs2 = f2_bcast(rstd);
      if constexpr (HEADS == 8) {
        uint32_t u[32];
        tmem_ld32(tmem + TM_D, u);
#pragma unroll
        for (int c = 0; c < 16; ++c) t[c] = ffma2(make_float2(__uint_as_float(u[2 * c]), __uint_as_float(u[2 * c + 1])), rs2, cA2[c]);
      } else {
        uint32_t u[16];
        tmem_ld16(tmem + TM_D, u);
#pragma unroll
        for (int c = 0; c < 8; ++c) t[c] = ffma2(make_float2(__uint_as_float(u[2 * c]), __uint_as_float(u[2 * c + 1])), rs2, cA2[c]);
#pragma unroll
        for (int c = 8; c < 16; ++c) t[c] = make_float2(0.f, 0.f);
      }
      turn_wait();
#pragma unroll
      for (int h = 0; h < HEADS; ++h) {                          // scores are in log2 units (tables kernel): 2^(s - max)
        const float2 a = t[2 * h], b = t[2 * h + 1];
        const float2 nmx = f2_bcast(-fmaxf(fmaxf(a.x, a.y), fmaxf(b.x, b.y)));
        const float2 da = fadd2(a, nmx), db = fadd2(b, nmx);
        const float2 ea = make_float2(ex2_approx(da.x), ex2_approx(da.y)), eb = make_float2(ex2_approx(db.x), ex2_approx(db.y));
        const float2 sm = fadd2(ea, eb);
        const float2 inv = f2_bcast(rcp_approx(sm.x + sm.y));
        t[2 * h] = fmul2(ea, inv); t[2 * h + 1] = fmul2(eb, inv);
      }
      write_a_row(t);
      turn_pass();
    }
    mma_round(t_hi + 4096, t_lo + 4096, IDESC_32, TM_X, KP{}, true);
    // ---- 3. Hid = xhat' . W1f^T        (Hid = rstd * ((x - mu) . W1f) + b1f)
    {
      uint32_t u[32];
      tmem_ld32(tmem + TM_X, u);
      turn_wait();
#pragma unroll
      for (int c = 0; c < 16; ++c) xr[c] = fadd2(make_float2(__uint_as_float(u[2 * c]), __uint_as_float(u[2 * c + 1])), cbA2[c]);
      rstd = center(xr, t);
      write_a_row(t);
      turn_pass();
    }
    mma_round(m_hi, m_lo, IDESC_32, TM_D, K4{}, false);
    // ---- 4. x += gelu(Hid + b1f) . W2^T
    {
      uint32_t u[32];
      tmem_ld32(tmem + TM_D, u);
      turn_wait();
      const float2 rs2 = f2_bcast(rstd);
#pragma unroll
      for (int c = 0; c < 16; ++c)
        t[c] = gelu_phi8_2(ffma2(make_float2(__uint_as_float(u[2 * c]), __uint_as_float(u[2 * c + 1])), rs2, b1f2[c]));
      write_a_row(t);
      turn_pass();
    }
    mma_round(m_hi + 4096, m_lo + 4096, IDESC_32, TM_X, K4{}, true);
    {
      uint32_t u[32];
      tmem_ld32(tmem + TM_X, u);
#pragma unroll
      for (int c = 0; c < 16; ++c) xr[c] = fadd2(make_float2(__uint_as_float(u[2 * c]), __uint_as_float(u[2 * c + 1])), cbM2[c]);
    }
    // this warpgroup is done with buffer b (its MMAs completed, its bias reads are in registers)
    asm volatile("bar.sync %0, 128;" ::"r"(wg + 1) : "memory");
    if (issuer) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&free_bar[b])) : "memory");
  }

#pragma unroll
  for (int q = 0; q < 8; ++q)
    *reinterpret_cast<float4*>(io + lane * 32 + ((q ^ (lane & 7)) << 2)) = make_float4(xr[q * 2].x, xr[q * 2].y, xr[q * 2 + 1].x, xr[q * 2 + 1].y);
  __syncwarp();
  if (out_split_plane || h16) {
    // split16 planes for conv_tc3.cu (hi = f16(o), lo = f16(2^11 (o - hi))), or h16: hi alone, and the skip is one FP16 plane
    // too: 4 lanes x 8 channels per pixel row, 16 bytes per lane and plane
    const int c4 = lane & 3, r4 = lane >> 2;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const int r = g * 8 + r4, pr = pw0 + r;
      if (pr < npix) {
        float4 o0 = *reinterpret_cast<const float4*>(io + r * 32 + (((2 * c4) ^ (r & 7)) << 2));
        float4 o1 = *reinterpret_cast<const float4*>(io + r * 32 + (((2 * c4 + 1) ^ (r & 7)) << 2));
        if (skip) {
          const int py = pr / w, px = pr - py * w;
          const size_t so = (skip_up == 2) ? (((size_t)img * (npix / w / 2) + (py >> 1)) * (w >> 1) + (px >> 1)) * 32
                                           : ((size_t)img * npix + pr) * 32;
          float4 v0, v1;
          if (h16) {
            const uint4 u = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(skip) + so + c4 * 8));
            v0 = make_float4(f16_lo(u.x), f16_hi(u.x), f16_lo(u.y), f16_hi(u.y));
            v1 = make_float4(f16_lo(u.z), f16_hi(u.z), f16_lo(u.w), f16_hi(u.w));
          } else {
            v0 = ldg4(skip + so + c4 * 8); v1 = ldg4(skip + so + c4 * 8 + 4);
          }
          o0.x += v0.x; o0.y += v0.y; o0.z += v0.z; o0.w += v0.w;
          o1.x += v1.x; o1.y += v1.y; o1.z += v1.z; o1.w += v1.w;
        }
        uint4 hi;
        hi.x = pack_f16x2_sat(o0.x, o0.y); hi.y = pack_f16x2_sat(o0.z, o0.w); hi.z = pack_f16x2_sat(o1.x, o1.y); hi.w = pack_f16x2_sat(o1.z, o1.w);
        uint16_t* o16 = reinterpret_cast<uint16_t*>(out);
        const size_t off = ((size_t)img * npix + pr) * 32 + c4 * 8;
        *reinterpret_cast<uint4*>(o16 + off) = hi;
        if (out_split_plane) {
          uint4 lo;
          lo.x = pack_f16x2_sat((o0.x - f16_lo(hi.x)) * 2048.f, (o0.y - f16_hi(hi.x)) * 2048.f);
          lo.y = pack_f16x2_sat((o0.z - f16_lo(hi.y)) * 2048.f, (o0.w - f16_hi(hi.y)) * 2048.f);
          lo.z = pack_f16x2_sat((o1.x - f16_lo(hi.z)) * 2048.f, (o1.y - f16_hi(hi.z)) * 2048.f);
          lo.w = pack_f16x2_sat((o1.z - f16_lo(hi.w)) * 2048.f, (o1.w - f16_hi(hi.w)) * 2048.f);
          *reinterpret_cast<uint4*>(o16 + off + (size_t)out_split_plane) = lo;
        }
      }
    }
  } else {
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      const int r = g * 4 + r8, pr = pw0 + r;
      if (pr < npix) {
        float4 o = *reinterpret_cast<const float4*>(io + r * 32 + ((c8 ^ (r & 7)) << 2));
        if (skip) {
          const int py = pr / w, px = pr - py * w;
          const float* sp = (skip_up == 2)
              ? skip + (((size_t)img * (npix / w / 2) + (py >> 1)) * (w >> 1) + (px >> 1)) * 32
              : skip + ((size_t)img * npix + pr) * 32;
          const float4 v = ldg4(sp + c8 * 4);
          o.x += v.x; o.y += v.y; o.z += v.z; o.w += v.w;
        }
        st4(out + ((size_t)img * npix + pr) * 32 + c8 * 4, o);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 32) {
    tc_fence_after();
    tmem_dealloc(tmem_slot, 512);
  }
}

template <int HEADS, bool X3>
int launch_pdt(dim3 grid, const float* x, const float* pos, const float* tables, const float* pack, int npix, int w, int depth,
               const float* skip, int skip_up, float* out, long long osp, int h16, cudaStream_t s) {
  cudaError_t e = cudaFuncSetAttribute(pixel_decoder_tc_kernel<HEADS, X3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)PdtCfg<X3>::SMEM);
  if (e != cudaSuccess) return (int)e;
  return dh_launch(pixel_decoder_tc_kernel<HEADS, X3>, grid, dim3(PDT_ROWS * PdtCfg<X3>::G), (size_t)PdtCfg<X3>::SMEM, s, x, pos, tables, pack,
                   npix, w, depth, skip, skip_up, out, (long long)osp, h16);
}
}  // namespace

int dh_launch_decoder_tables_tc(const float* mem, int B, int first_call, int ncalls, const float* dec, int heads, int depth,
                                float* tables, cudaStream_t s) {
  DH_REQUIRE(mem && dec && tables, DH_E_NULL);
  DH_REQUIRE(B > 0 && first_call >= 0 && ncalls >= 1 && first_call + ncalls <= 3 && (heads == 4 || heads == 8) && depth >= 1,
             DH_E_SHAPE);
  dim3 grid(depth, ncalls * B);
  const int smem = heads * 2048 * (int)sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(decoder_tables_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) return (int)e;
  return dh_launch(decoder_tables_tc_kernel, grid, dim3(128), (size_t)smem, s, mem, B, first_call, dec, heads, tables, depth);
}

// x3: bit 0 = error-compensated 3xTF32; bit 8 (x3 | 256): `out` receives split16 planes (conv_tc3.cu's input format);
// bit 9 (x3 | 512): x, skip and out are one FP16 plane each (the h16 mode)
int dh_launch_pixel_decoder_tc(const float* x, const float* pos, const float* tables, const float* pack, int nimg, int h,
                               int w, int heads, int depth, const float* skip, int skip_up, int x3, float* out,
                               cudaStream_t s) {
  const long long osp = (x3 & 256) ? (long long)nimg * h * w * 32 : 0;
  const int h16 = (x3 & 512) ? 1 : 0;
  DH_REQUIRE(!(h16 && osp), DH_E_VARIANT);
  x3 &= 1;
  DH_REQUIRE(x && tables && pack && out, DH_E_NULL);
  DH_REQUIRE(nimg > 0 && h > 0 && w > 0 && depth >= 1 && (heads == 4 || heads == 8), DH_E_SHAPE);
  DH_REQUIRE(!skip || skip_up == 1 || (skip_up == 2 && h % 2 == 0 && w % 2 == 0), DH_E_SHAPE);
  DH_REQUIRE(dh_aligned16(x) && dh_aligned16(pos) && dh_aligned16(tables) && dh_aligned16(pack) && dh_aligned16(skip) &&
             dh_aligned16(out), DH_E_ALIGN);
  const int npix = h * w;
  dim3 grid(dh_cdiv(npix, PDT_ROWS * PdtCfg<true>::G), nimg);
  if (heads == 4)
    return x3 ? launch_pdt<4, true>(grid, x, pos, tables, pack, npix, w, depth, skip, skip_up, out, osp, h16, s)
              : launch_pdt<4, false>(grid, x, pos, tables, pack, npix, w, depth, skip, skip_up, out, osp, h16, s);
  return x3 ? launch_pdt<8, true>(grid, x, pos, tables, pack, npix, w, depth, skip, skip_up, out, osp, h16, s)
            : launch_pdt<8, false>(grid, x, pos, tables, pack, npix, w, depth, skip, skip_up, out, osp, h16, s);
}
