// dahitra_b200 — classifier head: 3x3 pad-1 conv 32 -> NC (NC <= 8) + bias, NHWC fp32 in, NCHW logits out, fused uint8
// argmax (ties -> lowest class index like torch.argmax).  Reference: models/networks.py:1249,1355 and the harness argmax
// models/evaluator.py:89-92.
//
// Same arithmetic, in the same order, as classifier_kernel in conv_ffma.cu (fp32 FMA on CUDA cores: the output has 2-5
// channels, far below a tensor-core tile) — results are bit-identical — but the input halo is fetched by TMA:
//   * one box {16 ch, 40, 18, 1} per (tile, 16-channel half) over the NHWC tensor, zero-filled outside the image (= the
//     conv padding), SWIZZLE_64B so that the eight pixels a quarter-warp reads with one 128-bit load sit in eight
//     different 16-byte bank groups.  No per-element index arithmetic or cp.async address generation: that was 35 % of
//     the instructions the previous kernel issued (ncu: ALU pipe 36 %, FMA pipe 41 %, issue-active 66 %).
//   * persistent CTAs (two per SM) walk the tile list with a ring of two half-halo buffers: while the 4 compute warps work
//     on one half, a producer warp has the next one in flight (full / empty mbarriers).
// CTA tile = 32 x 16 pixels; thread (lx, g) owns the 4 vertically adjacent pixels (lx, 4g..4g+3), so each 128-bit halo
// read feeds up to 3 output rows and each filter read feeds 4 pixels.
// H16: the input is one FP16 plane (the h16 mode).  A 64-byte row then holds all 32 channels of a pixel, so one box
// {32 ch, 40, 18, 1} per tile (the same bytes and swizzle as one fp32 half); every 16-byte read is converted to eight
// fp32 values and summed with the same packed FFMA2 / scalar chains.
#include "tc_common.cuh"
#include <cstdlib>

using namespace dhtc;

namespace {
// The box is 40 pixels wide although the halo needs 34: with a row pitch that is a multiple of 8 pixels the swizzle term of a
// pixel, ((p >> 1) & 3), depends only on its column, so every thread precomputes its 12 chunk offsets once and the inner
// loop has no address arithmetic at all (the 6 extra columns cost 18 % more L2 -> SM bytes, no extra HBM traffic to speak of)
constexpr int CT_TW = 32, CT_TH = 16, CT_HW = 40, CT_HH = CT_TH + 2, CT_CH = 16;
constexpr uint32_t CT_HALF_BYTES = CT_HH * CT_HW * CT_CH * 4;        // 46080: one TMA box (a multiple of 1024)
constexpr uint32_t CT_BUF = CT_HALF_BYTES;
constexpr int CT_NBUF = 2;
constexpr int CT_THREADS = 160;                                      // 4 compute warps + 1 producer warp

template <int NC, bool H16>
__global__ void __launch_bounds__(CT_THREADS, 2)
classifier_tma_kernel(const __grid_constant__ CUtensorMap tmIn, int H, int W, int tilesX, int tilesY, int ntiles,
                      const float* __restrict__ w, const float* __restrict__ bias, float* __restrict__ logits,
                      unsigned char* __restrict__ amax) {
  constexpr int NPASS = H16 ? 1 : 2;                                  // boxes per tile
  constexpr int PCH = H16 ? 32 : CT_CH;                               // channels per box
  extern __shared__ uint8_t ct_raw[];
  __shared__ __align__(8) uint64_t full[CT_NBUF], empty[CT_NBUF];
  const uint32_t base = (smem_u32(ct_raw) + 1023u) & ~1023u;
  uint8_t* bp = ct_raw + (base - smem_u32(ct_raw));
  float* w_s = reinterpret_cast<float*>(bp + CT_NBUF * CT_BUF);        // [9][NC][32]
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) {
    for (int i = 0; i < CT_NBUF; ++i) { mbar_init(smem_u32(&full[i]), 1); mbar_init(smem_u32(&empty[i]), 4); }
    mbar_fence_init();
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmIn) : "memory");
  }
  for (int i = tid; i < 9 * NC * 8; i += CT_THREADS) reinterpret_cast<float4*>(w_s)[i] = __ldg(reinterpret_cast<const float4*>(w) + i);
  __syncthreads();
  dh_pdl_wait();                       // the input map comes from the previous launch (the filter above does not)
  dh_pdl_launch_dependents();

  if (warp == 4) {
    if ((tid & 31) == 0) {                                           // ---- producer: one box per (tile, half)
      int q = 0;
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int tx = tile % tilesX, ty = (tile / tilesX) % tilesY, n = tile / (tilesX * tilesY);
#pragma unroll
        for (int pass = 0; pass < NPASS; ++pass, ++q) {
          const int b = q % CT_NBUF;
          mbar_wait(smem_u32(&empty[b]), (uint32_t)(((q / CT_NBUF) & 1) ^ 1));
          mbar_expect_tx(smem_u32(&full[b]), CT_HALF_BYTES);
          tma_load_4d(base + (uint32_t)b * CT_BUF, &tmIn, smem_u32(&full[b]), pass * CT_CH, tx * CT_TW - 1, ty * CT_TH - 1, n);
        }
      }
    }
    return;
  }
  const int lx = tid & 31, g = tid >> 5;
  int choff[3][CT_CH / 4];                                 // float offset of chunk c4 inside the 16-channel row of column lx + s
#pragma unroll
  for (int s = 0; s < 3; ++s)
#pragma unroll
    for (int c4 = 0; c4 < CT_CH / 4; ++c4) choff[s][c4] = (lx + s) * CT_CH + ((c4 ^ (((lx + s) >> 1) & 3)) << 2);
  float bsv[NC];
#pragma unroll
  for (int k = 0; k < NC; ++k) bsv[k] = __ldg(bias + k);
  int q = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int tx = tile % tilesX, ty = (tile / tilesX) % tilesY, n = tile / (tilesX * tilesY);
    // NC >= 3 is bound by FMA issue (1440 FMAs per pixel at 5 classes against 128 bytes of input): the channel sum is kept as
    // two partial sums per class (even / odd channel of each pair), so that every pair of products is ONE packed FFMA2 whose
    // operands are the natural register pairs of the 128-bit halo / filter loads; the halves are added once per pixel.
    // NC <= 2 (HBM-bound) keeps the scalar chain, bit-identical to classifier_kernel in conv_ffma.cu.
    constexpr bool PACK = NC >= 3;
    float acc[4][NC];
    float2 acc2[PACK ? 4 : 1][PACK ? NC : 1];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int k = 0; k < NC; ++k) {
        acc[j][k] = bsv[k];
        if (PACK) acc2[j][k] = make_float2(bsv[k], 0.f);
      }
#pragma unroll 1
    for (int pass = 0; pass < NPASS; ++pass, ++q) {
      const int b = q % CT_NBUF;
      mbar_wait(smem_u32(&full[b]), (uint32_t)((q / CT_NBUF) & 1));
      const float* halo = reinterpret_cast<const float*>(bp + (size_t)b * CT_BUF);     // [18 x 40 pixels][16 ch], 64-byte rows, SWIZZLE_64B
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        // H16 at 7 / 8 classes: the full unroll spills (8 classes still spill 12 bytes at the 168-register cap of two CTAs per
        // SM, like the fp32 form); the network runs 2 and 5 classes
        constexpr int C4_UNROLL = (H16 && NC >= 7) ? 2 : 8;
#pragma unroll C4_UNROLL
        for (int c4 = 0; c4 < (H16 ? 8 : CT_CH / 4); ++c4) {     // 4-channel groups (H16: two per 16-byte chunk)
          float4 ww[3][NC];                                // the three filter rows of column s for these 4 channels
#pragma unroll
          for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int k = 0; k < NC; ++k)
              ww[r][k] = *reinterpret_cast<const float4*>(&w_s[((r * 3 + s) * NC + k) * 32 + pass * PCH + c4 * 4]);
#pragma unroll
          for (int hr = 0; hr < 6; ++hr) {                 // halo row 4g + hr feeds output rows j = hr - r, r = 0..2
            // halo pixel p = (4g + hr) * 40 + lx + s; SWIZZLE_64B puts its chunk c4 at c4 ^ ((p >> 1) & 3) = c4 ^ (((lx + s) >> 1) & 3)
            float4 v;
            if (H16) {                                     // the 16-byte chunk c4 / 2 holds 8 channels; this group is its half c4 & 1
              const int ch = (lx + s) * CT_CH + (((c4 >> 1) ^ (((lx + s) >> 1) & 3)) << 2);   // = choff[s][c4 >> 1]
              const uint2 u = reinterpret_cast<const uint2*>(&halo[(4 * g + hr) * (CT_HW * CT_CH) + ch])[c4 & 1];
              v = make_float4(f16_lo(u.x), f16_hi(u.x), f16_lo(u.y), f16_hi(u.y));
            } else {
              v = *reinterpret_cast<const float4*>(&halo[(4 * g + hr) * (CT_HW * CT_CH) + choff[s][c4]]);
            }
#pragma unroll
            for (int r = 0; r < 3; ++r) {
              const int j = hr - r;
              if (j < 0 || j > 3) continue;
#pragma unroll
              for (int k = 0; k < NC; ++k) {
                if (PACK) {
                  acc2[j][k] = ffma2(make_float2(v.x, v.y), make_float2(ww[r][k].x, ww[r][k].y), acc2[j][k]);
                  acc2[j][k] = ffma2(make_float2(v.z, v.w), make_float2(ww[r][k].z, ww[r][k].w), acc2[j][k]);
                } else {
                  acc[j][k] = fmaf(v.x, ww[r][k].x, acc[j][k]);
                  acc[j][k] = fmaf(v.y, ww[r][k].y, acc[j][k]);
                  acc[j][k] = fmaf(v.z, ww[r][k].z, acc[j][k]);
                  acc[j][k] = fmaf(v.w, ww[r][k].w, acc[j][k]);
                }
              }
            }
          }
        }
      }
      __syncwarp();
      if (lx == 0) mbar_arrive_local(smem_u32(&empty[b]));   // this warp has read everything it needs from the buffer
    }
    if (PACK) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int k = 0; k < NC; ++k) acc[j][k] = acc2[j][k].x + acc2[j][k].y;
    }
    const int x = tx * CT_TW + lx;
    if (x < W) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int y = ty * CT_TH + 4 * g + j;
        if (y >= H) break;
        int best = 0;
        float bv = acc[j][0];
#pragma unroll
        for (int k = 0; k < NC; ++k) {
          logits[(((size_t)n * NC + k) * H + y) * W + x] = acc[j][k];
          if (k > 0 && acc[j][k] > bv) { bv = acc[j][k]; best = k; }
        }
        if (amax) amax[((size_t)n * H + y) * W + x] = (unsigned char)best;
      }
    }
  }
}
}  // namespace

namespace {
template <bool H16>
int launch_classifier(const void* in, int N, int H, int W, int nc, const float* w, const float* b, float* logits,
                      unsigned char* amax, cudaStream_t s) {
  DH_REQUIRE(in && w && b && logits, DH_E_NULL);
  DH_REQUIRE(N > 0 && H > 0 && W > 0 && nc >= 1 && nc <= 8, DH_E_SHAPE);
  DH_REQUIRE(dh_aligned16(in) && dh_aligned16(w), DH_E_ALIGN);
  const int tx = dh_cdiv(W, CT_TW), ty = dh_cdiv(H, CT_TH);
  const int ntiles = tx * ty * N;
  CUtensorMap tm;
  {
    const unsigned long long eb = H16 ? 2ull : 4ull;                   // bytes per element
    const unsigned long long dims[4] = {32ull, (unsigned long long)W, (unsigned long long)H, (unsigned long long)N};
    const unsigned long long strides[3] = {32 * eb, (unsigned long long)W * 32 * eb, (unsigned long long)H * W * 32 * eb};
    const unsigned box[4] = {H16 ? 32u : (unsigned)CT_CH, (unsigned)CT_HW, (unsigned)CT_HH, 1u};
    const int rc = H16 ? dh_encode_tiled_f16_sw(&tm, in, 4, dims, strides, box, 64) : dh_encode_tiled_f32_sw(&tm, in, 4, dims, strides, box, 64);
    if (rc) return rc;
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  dim3 grid((unsigned)(ntiles < 2 * sms ? ntiles : 2 * sms), 1, 1);       // persistent: two CTAs per SM
#define DH_CLS_CASE(NC)                                                                                                 \
  case NC: {                                                                                                            \
    const int smem = (int)(CT_NBUF * CT_BUF + 9 * NC * 32 * sizeof(float) + 1024);                                      \
    cudaError_t e = cudaFuncSetAttribute(classifier_tma_kernel<NC, H16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); \
    if (e != cudaSuccess) return (int)e;                                                                                \
    return dh_launch(classifier_tma_kernel<NC, H16>, grid, dim3(CT_THREADS), (size_t)smem, s, tm, H, W, tx, ty, ntiles, w, b, logits, amax); \
  }
  switch (nc) {
    DH_CLS_CASE(1) DH_CLS_CASE(2) DH_CLS_CASE(3) DH_CLS_CASE(4)
    DH_CLS_CASE(5) DH_CLS_CASE(6) DH_CLS_CASE(7) DH_CLS_CASE(8)
  }
#undef DH_CLS_CASE
  return DH_E_SHAPE;
}
}  // namespace

int dh_launch_classifier_tma(const float* in, int N, int H, int W, int nc, const float* w, const float* b,
                             float* logits, unsigned char* amax, cudaStream_t s) {
  return launch_classifier<false>(in, N, H, W, nc, w, b, logits, amax, s);
}
int dh_launch_classifier_h16(const void* in, int N, int H, int W, int nc, const float* w, const float* b,
                             float* logits, unsigned char* amax, cudaStream_t s) {
  return launch_classifier<true>(in, N, H, W, nc, w, b, logits, amax, s);
}
