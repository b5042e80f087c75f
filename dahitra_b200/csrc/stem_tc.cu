// dahitra_b200 — stem (7x7 stride-2 pad-3 conv 3 -> 64 + folded BN + ReLU) on the tensor cores.
//
// Replaces resnet.conv1 + bn1 + relu (reference models/networks.py:1120-1122, models/resnet.py:150-153).
// GEMM view: D[128 pixels][64] = A[128][K] . Wt[64][K]^T.  C_in = 3 cannot feed a TMA/UMMA row directly, so the im2col
// rows are assembled ON CHIP from a planar (NCHW) halo.  K is ordered (ci, r, s8): one zero-weight pad (the TMA box must
// start on a 16-byte boundary, one column left of the first tap) plus the 7 taps of one filter row of one channel
// = 8 CONSECUTIVE halo floats = four 8-byte shared-memory loads and two 16-byte stores
// into the K-major SWIZZLE_128B A tile, with no index table.  K = 21 groups x 8 = 168, padded to 192 = 6 K steps of 32.
//
// Persistent kernel, one CTA per SM, 13 warps:
//   warps 0-3 / 4-7  two builder warpgroups; thread t of each owns pixel t of the 8x16 tile.  Group 0 builds the even
//                    K steps into A buffer 0, group 1 the odd ones into buffer 1, so two steps are always in flight
//                    (a single builder warp per scheduler is issue-latency bound).
//   warps 8-11       epilogue: drain the accumulator of the previous tile (two TMEM accumulators), bias + ReLU, NHWC stores.
//   warp 12          one lane issues the tcgen05.mma's in K order as the A buffers fill (mbarriers a_full / a_free).
//   warp 13          one lane fetches the 3 x 21 x 40 input halo of the next tile with ONE TMA box over the NCHW tensor
//                    (no swizzle: the box lands as the planar [ci][row][40] halo; out-of-image pixels are zero-filled =
//                    the conv padding; the only HBM read), double-buffered through halo_full / halo_free.
// The filter image (pre-swizzled, 6 K-step tiles of 64x32; hi [+ lo]) is loaded once per CTA by one bulk copy.
// X3: error-compensated 3xTF32 — A rows are written as TF32 hi + lo tiles, the filter comes pre-split.
// The default fp32-grade mode runs stem_f16_kernel below (folded FP16 operands) instead.
#include "tc_common.cuh"

using namespace dhtc;

namespace {
constexpr int SK_TH = 8, SK_TW = 16;                 // output patch
constexpr int SK_HR = 2 * SK_TH + 5;                 // 21 halo rows
constexpr int SK_HCP = 40;                           // halo cols fetched (37 needed; 8-float groups read up to col 37)
constexpr int SK_PLANE = SK_HR * SK_HCP;             // 840 floats per channel
constexpr int SK_KSTEPS = 6;                         // 192 / 32
constexpr int SK_GROUPS = 21;                        // (ci, r) groups that carry data
constexpr uint32_t SK_A_BYTES = 128 * 128;           // one A tile
constexpr uint32_t SK_B_BYTES = SK_KSTEPS * 64 * 128;    // 48 KB filter image
constexpr uint32_t SK_HALO_BYTES = 3 * SK_PLANE * 4; // 10080 (one TMA box)
constexpr uint32_t SK_HALO_STRIDE = 10112;           // 128-byte aligned buffer pitch (TMA destination alignment)
constexpr uint32_t SK_IDESC = umma_idesc_tf32(128, 64);
constexpr int SK_THREADS = 14 * 32;

template <bool X3> struct SkCfg {
  static constexpr uint32_t NA = X3 ? 4 : 2;                      // A tiles: [buf0 hi, buf1 hi, buf0 lo, buf1 lo]
  static constexpr uint32_t NB = X3 ? 2 : 1;                      // filter images: hi (+ lo)
  static constexpr uint32_t OFF_B = NA * SK_A_BYTES;
  static constexpr uint32_t OFF_H = OFF_B + NB * SK_B_BYTES;      // two halo buffers
  static constexpr uint32_t OFF_E = OFF_H + 2 * SK_HALO_STRIDE;   // epilogue staging: 4 warps x 4 KB (offset is a multiple of 16)
  static constexpr uint32_t SMEM = OFF_E + 4 * 4096 + 1024;
};

__device__ __forceinline__ float sk_tf32(float v) { return tf32_round(v); }

struct SkTile { int n, oy0, ox0; };
__device__ __forceinline__ SkTile sk_tile(int t, int tilesX, int tilesY) {
  SkTile r;
  r.ox0 = (t % tilesX) * SK_TW; t /= tilesX;
  r.oy0 = (t % tilesY) * SK_TH;
  r.n = t / tilesY;
  return r;
}

// Halo producer (one lane): ONE TMA box per tile over the NCHW tensor, double-buffered through halo_full / halo_free.
// x start must be 16-byte aligned: the box starts one column left of the first tap.
// Images 0..nfirst-1 come from tmX, the rest from tmX2 (the pre / post image sets of one forward in ONE launch).
__device__ __forceinline__ void sk_halo_producer(const CUtensorMap* tmX, uint32_t halo_addr, uint64_t* halo_full, uint64_t* halo_free,
                                                 int tilesX, int tilesY, int ntiles, const CUtensorMap* tmX2 = nullptr, int nfirst = 1 << 30) {
  int it = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
    const int hb = it & 1;
    if (it >= 2) mbar_wait(smem_u32(&halo_free[hb]), (uint32_t)(((it >> 1) - 1) & 1));   // all builders left this buffer
    const SkTile tl = sk_tile(tile, tilesX, tilesY);
    const uint32_t bar = smem_u32(&halo_full[hb]);
    mbar_expect_tx(bar, SK_HALO_BYTES);
    const bool second = tl.n >= nfirst;
    tma_load_4d(halo_addr + (uint32_t)hb * SK_HALO_STRIDE, second ? tmX2 : tmX, bar, 2 * tl.ox0 - 4, 2 * tl.oy0 - 3, 0, second ? tl.n - nfirst : tl.n);
  }
}

// Epilogue of one 32-column slice of one warp's 32 accumulator rows: through a per-warp shared-memory transpose so that
// each store instruction writes four whole 128-byte lines (8 lanes per pixel) instead of 16 bytes of 32 different
// lines (same scheme as conv_tc2.cu); + bias, ReLU, NHWC.
__device__ __forceinline__ void sk_store_slice(const float (&v)[32], float* stage, int lane, int q, int j, const SkTile& t,
                                               int OH, int OW, const float* __restrict__ bias, float* __restrict__ out,
                                               long long split_plane = 0) {
  const int c4 = lane & 3, r4 = lane >> 2;              // lane -> (8-channel group, row within a group of 8): 16 bytes per lane and plane
#pragma unroll
  for (int k4 = 0; k4 < 8; ++k4)
    *reinterpret_cast<float4*>(stage + lane * 32 + ((k4 ^ (lane & 7)) << 2)) = make_float4(v[k4 * 4], v[k4 * 4 + 1], v[k4 * 4 + 2], v[k4 * 4 + 3]);
  __syncwarp();
  const float4 b0 = ldg4(bias + j * 32 + c4 * 8), b1 = ldg4(bias + j * 32 + c4 * 8 + 4);
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const int r = g * 8 + r4, mm = q * 32 + r;             // tile pixel (py = mm / 16, px = mm % 16)
    const int oy = t.oy0 + mm / SK_TW, ox = t.ox0 + mm % SK_TW;
    const float4 o0 = *reinterpret_cast<const float4*>(stage + r * 32 + (((2 * c4) ^ (r & 7)) << 2));
    const float4 o1 = *reinterpret_cast<const float4*>(stage + r * 32 + (((2 * c4 + 1) ^ (r & 7)) << 2));
    if (oy < OH && ox < OW) {
      const float4 r0 = make_float4(fmaxf(o0.x + b0.x, 0.f), fmaxf(o0.y + b0.y, 0.f), fmaxf(o0.z + b0.z, 0.f), fmaxf(o0.w + b0.w, 0.f));
      const float4 r1 = make_float4(fmaxf(o1.x + b1.x, 0.f), fmaxf(o1.y + b1.y, 0.f), fmaxf(o1.z + b1.z, 0.f), fmaxf(o1.w + b1.w, 0.f));
      const size_t off = ((size_t)(t.n * OH + oy) * OW + ox) * 64 + j * 32 + c4 * 8;
      if (split_plane < 0) {             // one FP16 plane (h16 mode)
        uint4 hi;
        hi.x = pack_f16x2_sat(r0.x, r0.y); hi.y = pack_f16x2_sat(r0.z, r0.w); hi.z = pack_f16x2_sat(r1.x, r1.y); hi.w = pack_f16x2_sat(r1.z, r1.w);
        *reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(out) + off) = hi;
      } else if (split_plane) {          // split16 planes for conv_tc3.cu: hi = f16(r), lo = f16(2^11 (r - hi))
        uint4 hi, lo;
        hi.x = pack_f16x2_sat(r0.x, r0.y); hi.y = pack_f16x2_sat(r0.z, r0.w); hi.z = pack_f16x2_sat(r1.x, r1.y); hi.w = pack_f16x2_sat(r1.z, r1.w);
        lo.x = pack_f16x2_sat((r0.x - f16_lo(hi.x)) * 2048.f, (r0.y - f16_hi(hi.x)) * 2048.f);
        lo.y = pack_f16x2_sat((r0.z - f16_lo(hi.y)) * 2048.f, (r0.w - f16_hi(hi.y)) * 2048.f);
        lo.z = pack_f16x2_sat((r1.x - f16_lo(hi.z)) * 2048.f, (r1.y - f16_hi(hi.z)) * 2048.f);
        lo.w = pack_f16x2_sat((r1.z - f16_lo(hi.w)) * 2048.f, (r1.w - f16_hi(hi.w)) * 2048.f);
        uint16_t* o16 = reinterpret_cast<uint16_t*>(out);
        *reinterpret_cast<uint4*>(o16 + off) = hi;
        *reinterpret_cast<uint4*>(o16 + off + (size_t)split_plane) = lo;
      } else {
        st4(out + off, r0); st4(out + off + 4, r1);
      }
    }
  }
  __syncwarp();
}

template <bool X3>
__global__ void __launch_bounds__(SK_THREADS, 1)
stem_tc_kernel(const __grid_constant__ CUtensorMap tmX, int OH, int OW, int tilesX, int tilesY, int ntiles,
               const float* __restrict__ wtc, const float* __restrict__ bias, float* __restrict__ out) {
  using Cfg = SkCfg<X3>;
  extern __shared__ uint8_t sk_raw[];
  __shared__ __align__(8) uint64_t w_bar, a_full[2], a_free[2], acc_full[2], acc_empty[2], halo_full[2], halo_free[2];
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t base = (smem_u32(sk_raw) + 1023u) & ~1023u;
  uint8_t* bp = sk_raw + (base - smem_u32(sk_raw));
  constexpr uint32_t A_LO = 2 * SK_A_BYTES;                            // lo twins of the two A tiles (X3)
  const uint32_t b_addr = base + Cfg::OFF_B;

  if (tid == 0) {
    mbar_init(smem_u32(&w_bar), 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&a_full[i]), 128);
      mbar_init(smem_u32(&a_free[i]), 1);
      mbar_init(smem_u32(&acc_full[i]), 1);
      mbar_init(smem_u32(&acc_empty[i]), 128);
      mbar_init(smem_u32(&halo_full[i]), 1);
      mbar_init(smem_u32(&halo_free[i]), 256);
    }
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(&tmem_slot), 128);               // two 64-column accumulators
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  if (warp < 8) {
    // ------------------------------------------------------------------ builders: two warpgroups
    const int wg = warp >> 2, t = tid & 127;                           // t = pixel of the tile
    const int py = t / SK_TW, px = t % SK_TW;
    const int pbase = (2 * py) * SK_HCP + 2 * px;                     // even: every 8-float group is 8-byte aligned
    const int swz = t & 7;
    int it = 0, use = 0;                                               // tiles done by this CTA; uses of this group's A buffer
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const int hb = it & 1;
      mbar_wait(smem_u32(&halo_full[hb]), (uint32_t)((it >> 1) & 1)); // this tile's halo has landed
      const float* halo = reinterpret_cast<const float*>(bp + Cfg::OFF_H + (size_t)hb * SK_HALO_STRIDE) + pbase;
      float* at = reinterpret_cast<float*>(bp + (size_t)wg * SK_A_BYTES) + t * 32;
#pragma unroll 1
      for (int kt = wg; kt < SK_KSTEPS; kt += 2, ++use) {
        if (use >= 1) mbar_wait(smem_u32(&a_free[wg]), (uint32_t)((use - 1) & 1));   // the MMAs that read this buffer are done
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int g = kt * 4 + j;                                    // (ci, r) group; groups 21..23 are K padding
          float v[8];
          if (g < SK_GROUPS) {
            const float2* src = reinterpret_cast<const float2*>(halo + (g / 7) * SK_PLANE + (g % 7) * SK_HCP);
#pragma unroll
            for (int q = 0; q < 4; ++q) { const float2 f = src[q]; v[2 * q] = f.x; v[2 * q + 1] = f.y; }
          } else {
#pragma unroll
            for (int q = 0; q < 8; ++q) v[q] = 0.f;
          }
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            const int o = ((2 * j + c) ^ swz) << 2;
            const float h0 = sk_tf32(v[c * 4]), h1 = sk_tf32(v[c * 4 + 1]), h2 = sk_tf32(v[c * 4 + 2]), h3 = sk_tf32(v[c * 4 + 3]);
            *reinterpret_cast<float4*>(at + o) = make_float4(h0, h1, h2, h3);
            if (X3) *reinterpret_cast<float4*>(at + A_LO / 4 + o) = make_float4(sk_tf32(v[c * 4] - h0), sk_tf32(v[c * 4 + 1] - h1),
                                                                              sk_tf32(v[c * 4 + 2] - h2), sk_tf32(v[c * 4 + 3] - h3));
          }
        }
        fence_async_smem();
        mbar_arrive_local(smem_u32(&a_full[wg]));
      }
      mbar_arrive_local(smem_u32(&halo_free[hb]));                     // this thread's reads of the halo are done
    }
  } else if (warp < 12) {
    // ------------------------------------------------------------------ epilogue warps 8..11
    const int q = warp & 3, lane = tid & 31;
    float* stage = reinterpret_cast<float*>(bp + Cfg::OFF_E + (size_t)q * 4096);
    int it = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const SkTile t = sk_tile(tile, tilesX, tilesY);
      const int ab = it & 1;
      mbar_wait(smem_u32(&acc_full[ab]), (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      const uint32_t tm = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)ab * 64;
#pragma unroll 1
      for (int j = 0; j < 2; ++j) {
        uint32_t u[32];
        float v[32];
        tmem_ld32(tm + (uint32_t)(j * 32), u);
        if (j == 1) {
          tc_fence_before();
          mbar_arrive_local(smem_u32(&acc_empty[ab]));
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(u[i]);
        sk_store_slice(v, stage, lane, q, j, t, OH, OW, bias, out);
      }
    }
  } else if (warp == 13) {
    // ------------------------------------------------------------------ halo producer (warp 13, one lane)
    if ((tid & 31) == 0) sk_halo_producer(&tmX, base + Cfg::OFF_H, halo_full, halo_free, tilesX, tilesY, ntiles);
  } else if ((tid & 31) == 0) {
    // ------------------------------------------------------------------ MMA issuer (warp 12, one lane)
    mbar_expect_tx(smem_u32(&w_bar), Cfg::NB * SK_B_BYTES);
    bulk_load_1d(b_addr, wtc, SK_B_BYTES, smem_u32(&w_bar));
    if (X3) bulk_load_1d(b_addr + SK_B_BYTES, wtc + SK_B_BYTES / 4, SK_B_BYTES, smem_u32(&w_bar));
    mbar_wait(smem_u32(&w_bar), 0);
    int it = 0;
    uint32_t full_phase[2] = {0, 0};
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const int ab = it & 1;
      mbar_wait(smem_u32(&acc_empty[ab]), (uint32_t)(((it >> 1) & 1) ^ 1));    // the epilogue drained this accumulator
      tc_fence_after();
      const uint32_t d = tmem_base + (uint32_t)ab * 64;
#pragma unroll
      for (int kt = 0; kt < SK_KSTEPS; ++kt) {
        const int buf = kt & 1;
        mbar_wait(smem_u32(&a_full[buf]), full_phase[buf]);
        full_phase[buf] ^= 1u;
        tc_fence_after();
        const uint32_t a_addr = base + (uint32_t)buf * SK_A_BYTES;
        const uint64_t ad = umma_desc_sw128(a_addr), bd = umma_desc_sw128(b_addr + (uint32_t)kt * 64 * 128);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_tf32(d, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), SK_IDESC, (kt | k) ? 1u : 0u);
        if (X3) {
          const uint64_t al = umma_desc_sw128(a_addr + A_LO), bl = umma_desc_sw128(b_addr + SK_B_BYTES + (uint32_t)kt * 64 * 128);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_tf32(d, al + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), SK_IDESC, 1u);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_tf32(d, ad + (uint64_t)(2 * k), bl + (uint64_t)(2 * k), SK_IDESC, 1u);
        }
        umma_commit(smem_u32(&a_free[buf]));
      }
      umma_commit(smem_u32(&acc_full[ab]));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 128);
  }
}
// ------------------------------------------------------------------------------------------------------------------
// Folded FP16 stem (mode 2; the default fp32-grade mode): the same on-chip im2col, 16-bit operands.
//   a.w ~= f16(a).f16(w) + f16(a).r_w + r_a.bf16(w),   r_w = w - f16(w),  r_a = a - f16(a)
// as in conv_tc2.cu's folded mode: ONE N = 128 FP16 MMA on the filter image [f16(w) ; f16(2^11 r_w)] gives the main
// product (accumulator columns 0..63) and the scaled filter-remainder product (columns 64..127); a N = 64 BF16 MMA adds
// bf16(r_a).bf16(w) onto columns 0..63; the epilogue returns col[c] + 2^-11 col[64 + c].  A K step is one 128-byte
// row of 16-bit values = 64 K elements = 8 (ci, r) groups: 3 K steps per tile (21 groups + 3 pad groups; the last
// step issues 3 of its 4 K = 16 MMAs).  Against the 3xTF32 form this halves the bytes the builders write and cuts the
// operand bytes the MMAs read from shared memory by 2.5x — the shared-memory port is what bounds this kernel.
// Three A buffers [f16 hi | bf16 lo] form a ring over the global K-step sequence; the two builder warpgroups take
// alternate steps.
constexpr int SF_KSTEPS = 3;
constexpr int SF_NBUF = 3;
constexpr uint32_t SF_A_BUF = 2 * SK_A_BYTES;                        // hi + lo tiles of one step
constexpr uint32_t SF_BM_STEP = 128 * 128;                           // main filter tile of one step: 128 rows x 128 B
constexpr uint32_t SF_BC_STEP = 64 * 128;                            // correction filter tile (bf16 w)
constexpr uint32_t SF_BM_BYTES = SF_KSTEPS * SF_BM_STEP, SF_BC_BYTES = SF_KSTEPS * SF_BC_STEP;
constexpr uint32_t SF_OFF_B = SF_NBUF * SF_A_BUF;
constexpr uint32_t SF_OFF_H = SF_OFF_B + SF_BM_BYTES + SF_BC_BYTES;
constexpr uint32_t SF_OFF_E = SF_OFF_H + 2 * SK_HALO_STRIDE;
constexpr uint32_t SF_SMEM = SF_OFF_E + 4 * 4096 + 1024;
constexpr uint32_t SF_IDESC_MAIN = umma_idesc_f16(128, 128), SF_IDESC_CORR = umma_idesc_bf16(128, 64), SF_IDESC_ONE = umma_idesc_f16(128, 64);
constexpr size_t SF_IMAGE_OFFSET_FLOATS = 2 * (SK_B_BYTES / 4);      // the 16-bit images follow the TF32 [hi | lo] images in DH_W_STEM_WTC

template <bool FOLD>   // FOLD = false: single-pass FP16 operands (rows 0..63 of the same filter tiles, no remainder products)
__global__ void __launch_bounds__(SK_THREADS, 1)
stem_f16_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmX2, int nfirst, int OH, int OW, int tilesX,
                int tilesY, int ntiles, const float* __restrict__ wtc, const float* __restrict__ bias, float* __restrict__ out,
                long long split_plane) {
  extern __shared__ uint8_t sk_raw[];
  __shared__ __align__(8) uint64_t w_bar, a_full[SF_NBUF], a_free[SF_NBUF], acc_full[2], acc_empty[2], halo_full[2], halo_free[2];
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t base = (smem_u32(sk_raw) + 1023u) & ~1023u;
  uint8_t* bp = sk_raw + (base - smem_u32(sk_raw));
  const uint32_t b_addr = base + SF_OFF_B;

  if (tid == 0) {
    mbar_init(smem_u32(&w_bar), 1);
    for (int i = 0; i < SF_NBUF; ++i) {
      mbar_init(smem_u32(&a_full[i]), 128);
      mbar_init(smem_u32(&a_free[i]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&acc_full[i]), 1);
      mbar_init(smem_u32(&acc_empty[i]), 128);
      mbar_init(smem_u32(&halo_full[i]), 1);
      mbar_init(smem_u32(&halo_free[i]), 256);
    }
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc(smem_u32(&tmem_slot), 256);               // two 128-column accumulators [main | scaled remainder]
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  // barrier init and the TMEM allocation above overlap the previous launch's tail; the images (possibly written by the launch
  // just before: device-side normalisation) and the output buffer (possibly still read by it) are only touched after this
  dh_pdl_wait();
  dh_pdl_launch_dependents();

  if (warp < 8) {
    // ------------------------------------------------------------------ builders: two warpgroups, alternate global K steps
    const int wg = warp >> 2, t = tid & 127;
    const int py = t / SK_TW, px = t % SK_TW;
    const int pbase = (2 * py) * SK_HCP + 2 * px;
    const int swz = t & 7;
    int it = 0, c = wg, buf = wg, use = 0;                             // c = global step (3 per tile); buf = c % 3; use = c / 3
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const int hb = it & 1;
      mbar_wait(smem_u32(&halo_full[hb]), (uint32_t)((it >> 1) & 1));
      const float* halo = reinterpret_cast<const float*>(bp + SF_OFF_H + (size_t)hb * SK_HALO_STRIDE) + pbase;
#pragma unroll 1
      for (; c < SF_KSTEPS * (it + 1); c += 2) {
        const int kt = c - SF_KSTEPS * it;
        if (use >= 1) mbar_wait(smem_u32(&a_free[buf]), (uint32_t)((use - 1) & 1));   // the MMAs that read this buffer are done
        uint8_t* row = bp + (size_t)buf * SF_A_BUF + t * 128;
        const int ng = kt == 2 ? 6 : 8;                                // last step: groups 16..20 + one zero group (chunks 6, 7 are never read)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (j < ng) {
            const int g = kt * 8 + j;
            uint4 hi = make_uint4(0u, 0u, 0u, 0u), lo = hi;
            if (g < SK_GROUPS) {
              const float2* src = reinterpret_cast<const float2*>(halo + (g / 7) * SK_PLANE + (g % 7) * SK_HCP);
              const float2 f0 = src[0], f1 = src[1], f2 = src[2], f3 = src[3];
              hi.x = pack_f16x2_sat(f0.x, f0.y); hi.y = pack_f16x2_sat(f1.x, f1.y);
              hi.z = pack_f16x2_sat(f2.x, f2.y); hi.w = pack_f16x2_sat(f3.x, f3.y);
              lo.x = pack_bf16x2(f0.x - f16_lo(hi.x), f0.y - f16_hi(hi.x)); lo.y = pack_bf16x2(f1.x - f16_lo(hi.y), f1.y - f16_hi(hi.y));
              lo.z = pack_bf16x2(f2.x - f16_lo(hi.z), f2.y - f16_hi(hi.z)); lo.w = pack_bf16x2(f3.x - f16_lo(hi.w), f3.y - f16_hi(hi.w));
            }
            const int o = (j ^ swz) << 4;
            *reinterpret_cast<uint4*>(row + o) = hi;
            if (FOLD) *reinterpret_cast<uint4*>(row + SK_A_BYTES + o) = lo;
          }
        }
        fence_async_smem();
        mbar_arrive_local(smem_u32(&a_full[buf]));
        buf += 2;
        if (buf >= SF_NBUF) { buf -= SF_NBUF; ++use; }
      }
      mbar_arrive_local(smem_u32(&halo_free[hb]));
    }
  } else if (warp < 12) {
    // ------------------------------------------------------------------ epilogue warps 8..11: main + 2^-11 scaled remainder
    const int q = warp & 3, lane = tid & 31;
    float* stage = reinterpret_cast<float*>(bp + SF_OFF_E + (size_t)q * 4096);
    int it = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const SkTile t = sk_tile(tile, tilesX, tilesY);
      const int ab = it & 1;
      mbar_wait(smem_u32(&acc_full[ab]), (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      const uint32_t tm = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)ab * 128;
#pragma unroll 1
      for (int j = 0; j < 2; ++j) {
        uint32_t u[32], r[32];
        float v[32];
        tmem_ld32(tm + (uint32_t)(j * 32), u);
        if (FOLD) tmem_ld32(tm + (uint32_t)(64 + j * 32), r);
        if (j == 1) {
          tc_fence_before();
          mbar_arrive_local(smem_u32(&acc_empty[ab]));
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = FOLD ? fmaf(__uint_as_float(r[i]), 0x1p-11f, __uint_as_float(u[i])) : __uint_as_float(u[i]);
        sk_store_slice(v, stage, lane, q, j, t, OH, OW, bias, out, split_plane);
      }
    }
  } else if (warp == 13) {
    // ------------------------------------------------------------------ halo producer (warp 13, one lane)
    if ((tid & 31) == 0) sk_halo_producer(&tmX, base + SF_OFF_H, halo_full, halo_free, tilesX, tilesY, ntiles, &tmX2, nfirst);
  } else if ((tid & 31) == 0) {
    // ------------------------------------------------------------------ MMA issuer (warp 12, one lane)
    mbar_expect_tx(smem_u32(&w_bar), SF_BM_BYTES + SF_BC_BYTES);
    bulk_load_1d(b_addr, wtc + SF_IMAGE_OFFSET_FLOATS, SF_BM_BYTES, smem_u32(&w_bar));
    bulk_load_1d(b_addr + SF_BM_BYTES, wtc + SF_IMAGE_OFFSET_FLOATS + SF_BM_BYTES / 4, SF_BC_BYTES, smem_u32(&w_bar));
    mbar_wait(smem_u32(&w_bar), 0);
    int it = 0, buf = 0;
    uint32_t ph = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const int ab = it & 1;
      mbar_wait(smem_u32(&acc_empty[ab]), (uint32_t)(((it >> 1) & 1) ^ 1));
      tc_fence_after();
      const uint32_t d = tmem_base + (uint32_t)ab * 128;
#pragma unroll
      for (int kt = 0; kt < SF_KSTEPS; ++kt) {
        mbar_wait(smem_u32(&a_full[buf]), ph);
        tc_fence_after();
        const uint32_t a_addr = base + (uint32_t)buf * SF_A_BUF;
        const uint64_t ah = umma_desc_sw128(a_addr), al = umma_desc_sw128(a_addr + SK_A_BYTES);
        const uint64_t bm = umma_desc_sw128(b_addr + (uint32_t)kt * SF_BM_STEP);
        const uint64_t bc = umma_desc_sw128(b_addr + SF_BM_BYTES + (uint32_t)kt * SF_BC_STEP);
        constexpr int NK = 4;
#pragma unroll
        for (int k = 0; k < NK; ++k)
          if (kt < 2 || k < 3) umma_bf16(d, ah + (uint64_t)(2 * k), bm + (uint64_t)(2 * k), FOLD ? SF_IDESC_MAIN : SF_IDESC_ONE, (kt | k) ? 1u : 0u);
        if (FOLD) {
#pragma unroll
          for (int k = 0; k < NK; ++k)
            if (kt < 2 || k < 3) umma_bf16(d, al + (uint64_t)(2 * k), bc + (uint64_t)(2 * k), SF_IDESC_CORR, 1u);
        }
        umma_commit(smem_u32(&a_free[buf]));
        if (++buf == SF_NBUF) { buf = 0; ph ^= 1u; }
      }
      umma_commit(smem_u32(&acc_full[ab]));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}
}  // namespace

// x3: 0 = 1xTF32, 1 = 3xTF32, 2 = folded FP16, 3 = single-pass FP16; bit 8 (x3 | 256, modes 2 / 3 only): `out` receives the
// split16 planes conv_tc3.cu consumes instead of fp32; bit 9 (x3 | 512, mode 3 only): one FP16 plane (the h16 mode)
int dh_launch_stem_tc(const float* x, long long xbs, int N, int H, int W, const float* wtc, const float* b, float* out,
                      int x3, cudaStream_t s, long long split_plane_pitch, const float* x_second) {
  // x_second != NULL (forms 2 / 3): ONE launch over 2N images — N from x, then N from x_second (same strides) — writing one
  // [2N]-image output tensor: the pre and post image sets of a forward without a second launch
  const bool split = (x3 & 256) != 0, h16 = (x3 & 512) != 0;
  DH_REQUIRE(!(x3 & ~(255 | 256 | 512)) && !(split && h16), DH_E_VARIANT);
  x3 &= 255;
  DH_REQUIRE(!x_second || x3 == 2 || x3 == 3, DH_E_VARIANT);
  DH_REQUIRE(!split || x3 == 2 || x3 == 3, DH_E_VARIANT);
  DH_REQUIRE(!h16 || x3 == 3, DH_E_VARIANT);
  DH_REQUIRE(x && wtc && b && out, DH_E_NULL);
  DH_REQUIRE(N > 0 && H >= 8 && W >= 8 && H % 2 == 0 && W % 2 == 0, DH_E_SHAPE);
  DH_REQUIRE(dh_aligned16(wtc) && dh_aligned16(b) && dh_aligned16(out), DH_E_ALIGN);
  DH_REQUIRE((reinterpret_cast<uintptr_t>(x) & 3u) == 0, DH_E_ALIGN);
  const int OH = H / 2, OW = W / 2;
  const int tx = dh_cdiv(OW, SK_TW), ty = dh_cdiv(OH, SK_TH);
  const int nimg = x_second ? 2 * N : N;
  const int ntiles = tx * ty * nimg;
  // elements between the hi and lo planes: this call's own images, or the pitch of a larger tensor it writes a part of
  // (< 0: one FP16 plane)
  const long long split_plane = h16 ? -1 : split ? (split_plane_pitch ? split_plane_pitch : (long long)nimg * OH * OW * 64) : 0;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  dim3 grid((unsigned)(ntiles < sms ? ntiles : sms), 1, 1);
  DH_REQUIRE(W % 4 == 0 && xbs % 4 == 0 && dh_aligned16(x), DH_E_ALIGN);           // TMA: 16-byte global strides / base
  CUtensorMap tmX;                                                                  // NCHW input as (W, H, 3, N)
  {
    const unsigned long long dims[4] = {(unsigned long long)W, (unsigned long long)H, 3ull, (unsigned long long)N};
    const unsigned long long strides[3] = {(unsigned long long)W * 4, (unsigned long long)H * W * 4, (unsigned long long)xbs * 4};
    const unsigned box[4] = {(unsigned)SK_HCP, (unsigned)SK_HR, 3u, 1u};
    const int rc = dh_encode_tiled_f32(&tmX, x, 4, dims, strides, box, false);
    if (rc) return rc;
  }
  CUtensorMap tmX2 = tmX;
  if (x_second) {
    DH_REQUIRE(dh_aligned16(x_second), DH_E_ALIGN);
    const unsigned long long dims[4] = {(unsigned long long)W, (unsigned long long)H, 3ull, (unsigned long long)N};
    const unsigned long long strides[3] = {(unsigned long long)W * 4, (unsigned long long)H * W * 4, (unsigned long long)xbs * 4};
    const unsigned box[4] = {(unsigned)SK_HCP, (unsigned)SK_HR, 3u, 1u};
    const int rc = dh_encode_tiled_f32(&tmX2, x_second, 4, dims, strides, box, false);
    if (rc) return rc;
  }
  const int nfirst = x_second ? N : (1 << 30);
  if (x3 == 2) {
    cudaError_t e = cudaFuncSetAttribute(stem_f16_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SF_SMEM);
    if (e != cudaSuccess) return (int)e;
    return dh_launch(stem_f16_kernel<true>, grid, dim3(SK_THREADS), SF_SMEM, s, tmX, tmX2, nfirst, OH, OW, tx, ty, ntiles, wtc, b, out, split_plane);
  } else if (x3 == 3) {
    cudaError_t e = cudaFuncSetAttribute(stem_f16_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SF_SMEM);
    if (e != cudaSuccess) return (int)e;
    return dh_launch(stem_f16_kernel<false>, grid, dim3(SK_THREADS), SF_SMEM, s, tmX, tmX2, nfirst, OH, OW, tx, ty, ntiles, wtc, b, out, split_plane);
  } else if (x3) {
    cudaError_t e = cudaFuncSetAttribute(stem_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SkCfg<true>::SMEM);
    if (e != cudaSuccess) return (int)e;
    stem_tc_kernel<true><<<grid, SK_THREADS, SkCfg<true>::SMEM, s>>>(tmX, OH, OW, tx, ty, ntiles, wtc, b, out);
  } else {
    cudaError_t e = cudaFuncSetAttribute(stem_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SkCfg<false>::SMEM);
    if (e != cudaSuccess) return (int)e;
    stem_tc_kernel<false><<<grid, SK_THREADS, SkCfg<false>::SMEM, s>>>(tmX, OH, OW, tx, ty, ntiles, wtc, b, out);
  }
  DH_CHECK_LAUNCH();
  return 0;
}
