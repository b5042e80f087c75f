// dahitra_b200 — implicit-GEMM convolution on tcgen05 over PRE-SPLIT activations (the default fp32-grade mode).
//
// Storage format "split16" of an activation tensor [N][H][W][C]: two FP16 planes of the same shape,
//     hi = f16(a)  (round to nearest, saturating),   lo = f16(2^11 (a - hi))            a ~= hi + 2^-11 lo
// (4 bytes per element like fp32; 22 significant bits while a is in the normal FP16 range, absolute error <= 3e-11 below
// it).  Every producer epilogue writes this pair, so a consumer's TMA lands MMA operands directly: no fp32 halo, no
// splitter pass, no conversion warps (conv_tc2.cu pays one shared-memory pass per halo chunk for that).
// Filters come pre-split the same way: h_w = f16(w), l_w = f16(2^11 (w - h_w))   (planes 3 and 4 of the *_WT slots).
//
//   a.w = h_a.h_w + 2^-11 (h_a.l_w + l_a.h_w) + O(2^-22)
//
// Per (tap, 32-channel chunk, K = 16 step) two MMAs, all operands FP16, fp32 accumulation in tensor memory:
//   wide    [h_a] x [h_w ; l_w]   N = 2 NT   -> accumulator columns [0, NT) = main, [NT, 2 NT) = 2^11 x correction
//   narrow  [l_a] x [h_w]         N = NT     -> added onto columns [NT, 2 NT)      (B = the first NT rows of the wide tile)
// and the epilogue returns main + 2^-11 corr.  The filter ring therefore carries two 16-bit planes per tap (conv_tc2's
// folded mode: three), and the halo ring two 16-bit halos per chunk.
//
// Geometry as conv_tc2.cu: M tile = 16 x 8 output pixels of one image; per 32-channel chunk the (16+2) x (8+2) halo of
// each plane is fetched ONCE by a 4-D TMA box {32 ch, 10, 18, 1} (SWIZZLE_64B, zero fill outside the image = the conv
// padding) and serves all nine taps through shifted-window UMMA descriptors (start + (r*10+s) pixels, SBO = 10 pixels);
// stride 2 reads the four phase images with TMA element strides; persistent CTAs, two TMEM accumulators.
// Warp roles: 0 = halo TMA producer, 1 = TMEM alloc + MMA issuer, 6 = filter TMA producer, 2..5 and 7..10 = two epilogue
// warpgroups: group g drains accumulator g (the even / odd tiles of the CTA), so two epilogues are in flight under the main
// loop — the epilogue-heavy shapes (tokenizer squeeze, pixel-shuffle convs, residual + split16 stores) were bound by one.
//
// Epilogue outputs: fp32 NHWC (optionally as the pixel-shuffle scatter of the upsample convolutions) or split16 planes;
// the residual may be fp32 or split16.
//
// Single-plane form (P1, the h16 mode): activations are stored as ONE FP16 plane (hi alone, 2 bytes per element) and the
// filter contributes h_w alone.  Per chunk one halo box, per (tap, chunk, K = 16 step) one N = NT MMA [h_a] x [h_w], an
// accumulator of NT columns; the epilogue stores one FP16 plane (plain or pixel-shuffle) or fp32, and reads an FP16 residual.  TOK epilogue (1x1 squeeze convolution of the tokenizer, reference
// models/networks.py:1177-1189, 1273-1280): ReLU, store, and the per-tile online-softmax partials (m, s, t[32]) of the four
// semantic tokens — what squeeze_tokens_kernel (tokens.cu) computes on CUDA cores in the other modes.
#include "tc_common.cuh"
#include <cstdlib>
#include <mutex>
#include <unordered_map>

using namespace dhtc;

namespace {

constexpr int T3_TH = 16, T3_TW = 8;                    // output patch
constexpr int T3_HW = T3_TW + 2, T3_HH = T3_TH + 2;     // halo 10 x 18
constexpr uint32_t T3_PLANE = 11776;                    // one 16-bit halo (180 px x 64 B = 11520), padded to the 512-B swizzle period
constexpr uint32_t T3_HALO = 2 * T3_PLANE;              // hi + lo = 23552 (1024-aligned)
constexpr int T3_MAX_HB = 4;
enum { EPI_F32 = 0, EPI_SPLIT = 1, EPI_TOK = 2 };        // output: fp32 NHWC / pixel-shuffle | split16 planes | tokenizer (xs + partials)

struct T3Args {
  const float* bias;
  const void* res; void* out;
  const float* wtok; float* partials;                   // TOK epilogue
  long long res_plane, out_plane;                       // elements between the hi and lo planes of res / out
  int OH, OW, Cout, relu, tilesX, tilesY, cchunks0, cchunks, Cin, ps, N, ncout_tiles, ntiles;
  int res_split, out_split, tiles_per_img;
  int hb;                                               // halo buffers in use (2..T3_MAX_HB; what fits next to a resident filter)
  uint32_t halo_plane_bytes;                            // bytes one TMA box delivers (hw * hh * 64)
};

// RES = false: the filter tile of every (tap, chunk) streams from L2 through a TMA ring, once per M tile.
// RES = true:  the WHOLE filter ([ncout_tiles][cchunks][taps] tiles of [h_w ; l_w], <= 144 KB) is loaded into shared
//              memory once per CTA and stays there while the persistent CTA walks its tiles — the L2 -> SM path
//              (~43 B/clk per SM with every SM pulling, B300_MICROARCH "LTS throughput cap") is what bounds the
//              streaming form on the small-K layers: layer1 re-reads 144 KB of filter for every 46 KB halo.
template <int NT, bool RES, int CG = 1, bool P1 = false> struct T3Cfg {
  static constexpr int TPS = NT == 128 ? 1 : 3;                          // filter taps per ring stage (streaming form)
  static constexpr int STAGES = RES ? 1 : (NT == 128 ? 6 : (NT == 64 ? 4 : 8)) * CG;   // a CTA of a pair holds half-size tiles
  static constexpr uint32_t HALO = P1 ? T3_PLANE : T3_HALO;             // bytes of one halo buffer
  static constexpr uint32_t B_TAP = (P1 ? 1u : 2u) * NT * 64u / CG;      // [h_w ; l_w] (P1: h_w) x 64 B: NT rows each, NT / 2 in a CTA of a pair
  static constexpr uint32_t B_STAGE = B_TAP * TPS;
  static constexpr uint32_t RING_BYTES = RES ? 0u : STAGES * B_STAGE;    // RES: the filter image follows the halo buffers instead
  static constexpr int THREADS = 352;                                    // 11 warps: halo, MMA, epilogue A x4, filter, epilogue B x4
  static constexpr uint32_t IDESC_WIDE = umma_idesc_f16(128, 2 * NT);
  static constexpr uint32_t IDESC_NARROW = umma_idesc_f16(128 * CG, NT);
  static constexpr int ACC_COLS = P1 ? NT : 2 * NT;
  static constexpr uint32_t TMEM_COLS = 2 * ACC_COLS < 32 ? 32 : 2 * ACC_COLS;
};

template <int KS, int SD> struct Tap3 {                                   // tap order / halo shifts (see conv_tc2.cu TapSched)
  static constexpr int NPH = (KS == 3 && SD == 2) ? 4 : 1;
  static constexpr int NTAPS = KS * KS;
  __host__ __device__ static constexpr int tap(int i) {
    return (KS == 3 && SD == 2) ? (int)((0x862071534ULL >> (4 * i)) & 0xF) : i;   // stride 2: {4, 3,5, 1,7, 0,2,6,8} grouped by phase
  }
  __host__ __device__ static constexpr int first(int ph) {
    return (KS == 3 && SD == 2) ? (int)((0x95310u >> (4 * ph)) & 0xF) : (ph == 0 ? 0 : NTAPS);
  }
  __host__ __device__ static constexpr int shift_px(int t, int halo_w) {
    return KS == 1 ? 0 : (SD == 2 ? ((t / 3 != 0) ? halo_w : 0) + ((t % 3 != 0) ? 1 : 0) : (t / 3) * halo_w + t % 3);
  }
};

struct Tile3 { int n, oy0, ox0, ct; };
// CG = 2: work item = (pair of consecutive M tiles, cout tile); CTA `rank` of the pair takes M tile 2 * pair + rank.  The odd
// tile of the last pair may not exist: then n == e.N, its TMA boxes lie outside the tensor (zero fill) and its epilogue
// stores nothing.
__device__ __forceinline__ Tile3 tile3(int tile, const T3Args& e, int CG = 1, int rank = 0) {
  Tile3 t;
  t.ct = tile % e.ncout_tiles; tile /= e.ncout_tiles;
  if (CG == 2) tile = 2 * tile + rank;
  const int tx = tile % e.tilesX; tile /= e.tilesX;
  const int ty = tile % e.tilesY;
  t.n = tile / e.tilesY; t.oy0 = ty * T3_TH; t.ox0 = tx * T3_TW;
  return t;
}

// (pair) issued by either CTA, completion bytes counted on `cluster_bar` (the leader's barrier)
__device__ __forceinline__ void tma_load_3d_2sm(uint32_t dst, const CUtensorMap* tm, uint32_t cluster_bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(tm), "r"(cluster_bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// split16 pack / unpack of eight values (16 bytes per plane)
__device__ __forceinline__ void split8(const float4& a, const float4& b, uint4& hi, uint4& lo) {
  hi.x = pack_f16x2_sat(a.x, a.y); hi.y = pack_f16x2_sat(a.z, a.w); hi.z = pack_f16x2_sat(b.x, b.y); hi.w = pack_f16x2_sat(b.z, b.w);
  lo.x = pack_f16x2_sat((a.x - f16_lo(hi.x)) * 2048.f, (a.y - f16_hi(hi.x)) * 2048.f);
  lo.y = pack_f16x2_sat((a.z - f16_lo(hi.y)) * 2048.f, (a.w - f16_hi(hi.y)) * 2048.f);
  lo.z = pack_f16x2_sat((b.x - f16_lo(hi.z)) * 2048.f, (b.y - f16_hi(hi.z)) * 2048.f);
  lo.w = pack_f16x2_sat((b.z - f16_lo(hi.w)) * 2048.f, (b.w - f16_hi(hi.w)) * 2048.f);
}
__device__ __forceinline__ void join8(const uint4& hi, const uint4& lo, float4& a, float4& b) {
  constexpr float S = 1.0f / 2048.0f;
  a = make_float4(fmaf(f16_lo(lo.x), S, f16_lo(hi.x)), fmaf(f16_hi(lo.x), S, f16_hi(hi.x)),
                  fmaf(f16_lo(lo.y), S, f16_lo(hi.y)), fmaf(f16_hi(lo.y), S, f16_hi(hi.y)));
  b = make_float4(fmaf(f16_lo(lo.z), S, f16_lo(hi.z)), fmaf(f16_hi(lo.z), S, f16_hi(hi.z)),
                  fmaf(f16_lo(lo.w), S, f16_lo(hi.w)), fmaf(f16_hi(lo.w), S, f16_hi(hi.w)));
}
__device__ __forceinline__ void half8(const uint4& h, float4& a, float4& b) {     // eight FP16 values -> fp32
  a = make_float4(f16_lo(h.x), f16_hi(h.x), f16_lo(h.y), f16_hi(h.y));
  b = make_float4(f16_lo(h.z), f16_hi(h.z), f16_lo(h.w), f16_hi(h.w));
}
__device__ __forceinline__ uint4 ldg16(const void* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ float4 as_f4(const uint4& u) { return make_float4(__uint_as_float(u.x), __uint_as_float(u.y), __uint_as_float(u.z), __uint_as_float(u.w)); }

// CG = 2: CTA pairs (tcgen05 cta_group::2, cluster of two).  The leader (rank 0) issues M = 256 MMAs over both CTAs' halos;
// every B operand is split across the pair by N halves, so each CTA loads, stores and reads only half of every filter tile —
// half the L2 -> SM filter traffic and half the B reads from shared memory per pixel.  With B split by rows the N-doubled
// "wide" tile cannot be used (its two halves would need different partners), so the three partial products are issued as
// three N = NT MMAs: h_a.h_w -> main; h_a.l_w, l_a.h_w -> corr — the same tensor-core cycles as wide + narrow.
// Barriers the MMA warp waits on live in the leader and count both CTAs (the peer's TMA / threads signal them remotely);
// the leader's commits are multicast to both CTAs' barriers.
template <int NT, int KS, int SD, int EPI, bool RES, int CG, bool P1>
__global__ void __launch_bounds__(T3Cfg<NT, RES, CG, P1>::THREADS, 1)
conv_tc3_kernel(const __grid_constant__ CUtensorMap tmA0h, const __grid_constant__ CUtensorMap tmA0l,
                const __grid_constant__ CUtensorMap tmA1h, const __grid_constant__ CUtensorMap tmA1l,
                const __grid_constant__ CUtensorMap tmB, const T3Args e) {
  using Cfg = T3Cfg<NT, RES, CG, P1>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t t3_raw[];
  __shared__ __align__(8) uint64_t halo_full[T3_MAX_HB], halo_empty[T3_MAX_HB], b_full[STAGES], b_empty[STAGES], acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t base = (smem_u32(t3_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = t3_raw + (base - smem_u32(t3_raw));
  const int HB = e.hb;
  const uint32_t b_ring = base + (uint32_t)HB * Cfg::HALO;                 // filter ring, or the resident filter image
  const int rank = CG == 2 ? (int)cluster_ctarank() : 0;
  const int w0 = CG == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;      // first work item, and the stride between items
  const int wstep = CG == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  constexpr int pad = (KS == 3) ? 1 : 0;
  using Sched = Tap3<KS, SD>;
  constexpr int NPH = Sched::NPH;
  constexpr int NTAPS = KS * KS;
  constexpr int TPS = (SD == 1 && NTAPS % Cfg::TPS == 0) ? Cfg::TPS : 1;
  constexpr int HALO_W = (KS == 3) ? T3_HW : T3_TW;
  const uint32_t w_bytes = RES ? (uint32_t)(e.ncout_tiles * e.cchunks * NTAPS) * Cfg::B_TAP : Cfg::RING_BYTES;
  const uint32_t epi_off = (uint32_t)HB * Cfg::HALO + w_bytes;            // epilogue staging (8 warps x 4 KB), then the tok scratch

  if (threadIdx.x == 0) {
    for (int i = 0; i < T3_MAX_HB; ++i) { mbar_init(smem_u32(&halo_full[i]), 1); mbar_init(smem_u32(&halo_empty[i]), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(smem_u32(&acc_full[i]), 1); mbar_init(smem_u32(&acc_empty[i]), 128 * CG); }
    for (int s = 0; s < STAGES; ++s) { mbar_init(smem_u32(&b_full[s]), 1); mbar_init(smem_u32(&b_empty[s]), 1); }
    mbar_fence_init();
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA0h) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA0l) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
  }
  if (warp == 1) {
    if (CG == 2) tmem_alloc_2sm(smem_u32(&tmem_slot), Cfg::TMEM_COLS);
    else         tmem_alloc(smem_u32(&tmem_slot), Cfg::TMEM_COLS);
  }
  if (EPI == EPI_TOK && threadIdx.x >= 64 && threadIdx.x < 96)          // wtok [32][4] -> shared (weights: not produced by the previous launch)
    reinterpret_cast<float4*>(base_ptr + epi_off + 8 * 4096)[threadIdx.x - 64] = __ldg(reinterpret_cast<const float4*>(e.wtok) + (threadIdx.x - 64));
  tc_fence_before();
  __syncthreads();
  if (CG == 2) cluster_sync_all();                      // the peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  if (RES && warp == 6 && lane == 0) {
    // resident filter: every (cout tile, chunk, tap) tile, once (pair: this CTA's N half of each).  Weights are not written
    // by the previous launch, so this goes out before griddepcontrol.wait and overlaps that launch's tail under
    // programmatic dependent launch.
    const uint32_t bar = smem_u32(&b_full[0]);
    if (rank == 0) mbar_expect_tx(bar, (uint32_t)CG * w_bytes);             // pair: the leader's barrier counts both halves
    const uint32_t lbar = (CG == 2 && rank == 1) ? mapa_u32(bar, 0) : bar;
    uint32_t dst = b_ring;
    for (int ct = 0; ct < e.ncout_tiles; ++ct)
      for (int cc = 0; cc < e.cchunks; ++cc)
#pragma unroll
        for (int i = 0; i < NTAPS; ++i, dst += Cfg::B_TAP) {
          if (CG == 2) tma_load_3d_2sm(dst, &tmB, lbar, Sched::tap(i) * e.Cin + cc * 32, ct * NT + rank * (NT / 2), 0);
          else         tma_load_3d(dst, &tmB, bar, Sched::tap(i) * e.Cin + cc * 32, ct * NT, 0);
        }
  }
  // everything above overlaps the tail of the previous launch under programmatic dependent launch; its outputs (this
  // launch's activations / residual) are only touched below
  pdl_wait();
  pdl_launch_dependents();

  if (warp == 0) {
    if (lane == 0) {                                            // ---------------- halo TMA producer: hi + lo boxes per chunk (P1: hi)
      int hb = 0;
      uint32_t ephase = 1;                                      // first pass over the ring: the buffers are free
      for (int tile = w0; tile < e.ntiles; tile += wstep) {
        const Tile3 t = tile3(tile, e, CG, rank);
        for (int cc = 0; cc < e.cchunks; ++cc) {
#pragma unroll
          for (int ph = 0; ph < NPH; ++ph) {
            mbar_wait(smem_u32(&halo_empty[hb]), ephase);
            const uint32_t bar = smem_u32(&halo_full[hb]);
            if (rank == 0) mbar_expect_tx(bar, (uint32_t)CG * (P1 ? 1u : 2u) * e.halo_plane_bytes);   // pair: the leader's barrier counts both halos
            const uint32_t dst = base + (uint32_t)hb * Cfg::HALO;
            const int cx = SD == 1 ? t.ox0 - pad : 2 * (t.ox0 - pad) + (ph & 1);
            const int cy = SD == 1 ? t.oy0 - pad : 2 * (t.oy0 - pad) + (ph >> 1);
            const bool first = cc < e.cchunks0;
            const int c0 = (first ? cc : cc - e.cchunks0) * 32;
            if (CG == 2 && rank == 1) {
              const uint32_t lbar = mapa_u32(bar, 0);
              tma_load_4d_2sm(dst, first ? &tmA0h : &tmA1h, lbar, c0, cx, cy, t.n);
              tma_load_4d_2sm(dst + T3_PLANE, first ? &tmA0l : &tmA1l, lbar, c0, cx, cy, t.n);
            } else {
              tma_load_4d(dst, first ? &tmA0h : &tmA1h, bar, c0, cx, cy, t.n);
              if (!P1) tma_load_4d(dst + T3_PLANE, first ? &tmA0l : &tmA1l, bar, c0, cx, cy, t.n);
            }
            if (++hb == HB) { hb = 0; ephase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 6) {
    if (!RES && lane == 0) {                                    // ---------------- filter TMA producer: one 3-D box [2][NT][32] per tap
      int step = 0;
      for (int tile = w0; tile < e.ntiles; tile += wstep) {
        const Tile3 t = tile3(tile, e, CG, rank);
        for (int cc = 0; cc < e.cchunks; ++cc) {
#pragma unroll
          for (int i0 = 0; i0 < NTAPS; i0 += TPS, ++step) {
            const int st = step % STAGES, round = step / STAGES;
            mbar_wait(smem_u32(&b_empty[st]), (uint32_t)((round & 1) ^ 1));
            const uint32_t bar = smem_u32(&b_full[st]);
            if (rank == 0) mbar_expect_tx(bar, (uint32_t)(CG * TPS) * Cfg::B_TAP);          // pair: both halves
            const uint32_t lbar = (CG == 2 && rank == 1) ? mapa_u32(bar, 0) : bar;
#pragma unroll
            for (int tt = 0; tt < TPS; ++tt) {
              const uint32_t dst = b_ring + (uint32_t)st * Cfg::B_STAGE + (uint32_t)tt * Cfg::B_TAP;
              const int kcol = Sched::tap(i0 + tt) * e.Cin + cc * 32;
              if (CG == 2) tma_load_3d_2sm(dst, &tmB, lbar, kcol, t.ct * NT + rank * (NT / 2), 0);
              else         tma_load_3d(dst, &tmB, bar, kcol, t.ct * NT, 0);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {                               // ---------------- MMA issuer (pair: the leader only)
      constexpr uint32_t SBO = (uint32_t)HALO_W * 64u;
      int hb = 0, st = 0, it = 0;
      uint32_t hphase = 0, bphase = 0;
      if (RES) { mbar_wait(smem_u32(&b_full[0]), 0); tc_fence_after(); }     // the whole filter has landed
      for (int tile = w0; tile < e.ntiles; tile += wstep, ++it) {
        const int ab = it & 1;
        if (CG == 2) mbar_wait_cluster(smem_u32(&acc_empty[ab]), (uint32_t)(((it >> 1) & 1) ^ 1));
        else         mbar_wait(smem_u32(&acc_empty[ab]), (uint32_t)(((it >> 1) & 1) ^ 1));    // epilogue drained this accumulator
        tc_fence_after();
        const uint32_t d_main = tmem_base + (uint32_t)ab * Cfg::ACC_COLS, d_corr = d_main + NT;
        const uint32_t w_tile = RES ? b_ring + (uint32_t)((tile % e.ncout_tiles) * e.cchunks * NTAPS) * Cfg::B_TAP : 0u;
        for (int cc = 0; cc < e.cchunks; ++cc) {
#pragma unroll
          for (int ph = 0; ph < NPH; ++ph) {
            mbar_wait(smem_u32(&halo_full[hb]), hphase);
            tc_fence_after();
            const uint32_t h_hi = base + (uint32_t)hb * Cfg::HALO, h_lo = h_hi + T3_PLANE;
#pragma unroll
            for (int i0 = Sched::first(ph); i0 < Sched::first(ph + 1); i0 += TPS) {
              uint32_t b_stage;
              if (RES) {
                b_stage = w_tile + (uint32_t)(cc * NTAPS + i0) * Cfg::B_TAP;
              } else {
                mbar_wait(smem_u32(&b_full[st]), bphase);
                tc_fence_after();
                b_stage = b_ring + (uint32_t)st * Cfg::B_STAGE;
              }
#pragma unroll
              for (int tt = 0; tt < TPS; ++tt) {
                const int i = i0 + tt;
                const uint32_t px = (uint32_t)Sched::shift_px(Sched::tap(i), HALO_W) * 64u;      // compile-time after unrolling
                const uint64_t a_h = umma_desc_sw64(h_hi + px, SBO), a_l = umma_desc_sw64(h_lo + px, SBO);
                const uint64_t b_w = umma_desc_sw64(b_stage + (uint32_t)tt * Cfg::B_TAP, 512u);
                if (CG == 2) {
                  // this CTA's tile = [h_w half (NT/2 rows) ; l_w half]; the pair's halves form the N = NT operands
                  const uint64_t b_l = umma_desc_sw64(b_stage + (uint32_t)tt * Cfg::B_TAP + (NT / 2) * 64u, 512u);
#pragma unroll
                  for (int k = 0; k < 2; ++k) umma_bf16_2sm(d_main, a_h + (uint64_t)(2 * k), b_w + (uint64_t)(2 * k), Cfg::IDESC_NARROW, (cc | i | k) ? 1u : 0u);
#pragma unroll
                  for (int k = 0; k < 2; ++k) umma_bf16_2sm(d_corr, a_h + (uint64_t)(2 * k), b_l + (uint64_t)(2 * k), Cfg::IDESC_NARROW, (cc | i | k) ? 1u : 0u);
#pragma unroll
                  for (int k = 0; k < 2; ++k) umma_bf16_2sm(d_corr, a_l + (uint64_t)(2 * k), b_w + (uint64_t)(2 * k), Cfg::IDESC_NARROW, 1u);
                } else if (P1) {
#pragma unroll
                  for (int k = 0; k < 2; ++k) umma_bf16(d_main, a_h + (uint64_t)(2 * k), b_w + (uint64_t)(2 * k), Cfg::IDESC_NARROW, (cc | i | k) ? 1u : 0u);
                } else {
#pragma unroll
                  for (int k = 0; k < 2; ++k) umma_bf16(d_main, a_h + (uint64_t)(2 * k), b_w + (uint64_t)(2 * k), Cfg::IDESC_WIDE, (cc | i | k) ? 1u : 0u);
#pragma unroll
                  for (int k = 0; k < 2; ++k) umma_bf16(d_corr, a_l + (uint64_t)(2 * k), b_w + (uint64_t)(2 * k), Cfg::IDESC_NARROW, 1u);
                }
              }
              if (!RES) {
                if (CG == 2) umma_commit_2sm(smem_u32(&b_empty[st])); else umma_commit(smem_u32(&b_empty[st]));
                if (++st == STAGES) { st = 0; bphase ^= 1u; }
              }
            }
            if (CG == 2) umma_commit_2sm(smem_u32(&halo_empty[hb])); else umma_commit(smem_u32(&halo_empty[hb]));
            if (++hb == HB) { hb = 0; hphase ^= 1u; }
          }
        }
        if (CG == 2) umma_commit_2sm(smem_u32(&acc_full[ab])); else umma_commit(smem_u32(&acc_full[ab]));
      }
    }
  } else {                                                      // ---------------- epilogue (warps 2..5 = group 0, 7..10 = group 1)
    // Thread = accumulator row (pixel).  Every 32-channel slab goes through a per-warp shared-memory transpose so that the
    // global accesses are 4 lanes x 8 channels per pixel row: whole 128-byte lines of an fp32 tensor, 64-byte segments of
    // each split16 plane, 16 bytes per lane either way, 8 pixel rows per instruction.
    const int q = warp & 3, grp = warp >= 7 ? 1 : 0;            // q: the TMEM lane quarter this warp may read (warp id mod 4)
    float* stage = reinterpret_cast<float*>(base_ptr + epi_off + (size_t)(grp * 4 + q) * 4096);   // [32 rows][8 chunks ^ (row & 7)][4]
    const float* wtok_s = reinterpret_cast<const float*>(base_ptr + epi_off + 8 * 4096);          // [32][4]
    float* tokred = reinterpret_cast<float*>(base_ptr + epi_off + 8 * 4096 + 512 + grp * 2176);   // [4 warps][4 tokens][34] per group
    const int c4 = lane & 3, r4 = lane >> 2;                    // lane -> (8-channel group, row within a group of 8)
    constexpr int NSLAB = NT / 32;
    const char* resb = reinterpret_cast<const char*>(e.res);
    int it = 0;
    for (int tile = w0; tile < e.ntiles; tile += wstep, ++it) {
      if ((it & 1) != grp) continue;                             // this group owns accumulator `grp`
      const Tile3 t = tile3(tile, e, CG, rank);
      const int n0 = t.ct * NT;
      size_t rowoff[4];                                          // element offset of (pixel, channel group) for this lane's 4 rows
      bool ok[4];
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const int mm = q * 32 + g * 8 + r4;
        const int oy = t.oy0 + mm / T3_TW, ox = t.ox0 + mm % T3_TW;
        ok[g] = (oy < e.OH) && (ox < e.OW) && (t.n < e.N);
        rowoff[g] = e.ps ? ((size_t)(t.n * 2 * e.OH + 2 * oy) * (2 * e.OW) + 2 * ox) * 32 + c4 * 8
                         : ((size_t)(t.n * e.OH + oy) * e.OW + ox) * e.Cout + n0 + c4 * 8;
      }
      // residual of slab j: two 16-byte loads per row, raw (converted only when added, so that they stay in flight under
      // the accumulator wait, the TMEM loads and the transpose).  fp32: the two float4 of the 8 channels; split16: hi, lo.
      uint4 ra[4], rb[4];
      auto load_res = [&](int j) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          ra[g] = make_uint4(0u, 0u, 0u, 0u); rb[g] = ra[g];
          if (ok[g]) {
            const size_t o = rowoff[g] + (size_t)j * 32;
            if (e.res_split) { ra[g] = ldg16(resb + o * 2); if (!P1) rb[g] = ldg16(resb + (o + (size_t)e.res_plane) * 2); }
            else             { ra[g] = ldg16(resb + o * 4); rb[g] = ldg16(resb + o * 4 + 16); }
          }
        }
      };
      if (e.res) load_res(0);
      const int ab = it & 1;
      mbar_wait(smem_u32(&acc_full[ab]), (uint32_t)((it >> 1) & 1));
      tc_fence_after();
#pragma unroll 1
      for (int j = 0; j < NSLAB; ++j) {
        float4 bia0 = make_float4(0.f, 0.f, 0.f, 0.f), bia1 = bia0;
        if (e.bias) { bia0 = ldg4(e.bias + n0 + j * 32 + c4 * 8); bia1 = ldg4(e.bias + n0 + j * 32 + c4 * 8 + 4); }
        uint32_t v[32], u[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * Cfg::ACC_COLS + j * 32), v);
        if (!P1) tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * Cfg::ACC_COLS + NT + j * 32), u);
        if (j == NSLAB - 1) {                                    // accumulator fully read: hand it back to the MMA warp
          tc_fence_before();
          if (CG == 2) mbar_arrive_cluster(mapa_u32(smem_u32(&acc_empty[ab]), 0));
          else         mbar_arrive_local(smem_u32(&acc_empty[ab]));
        }
        float tl[4] = {0.f, 0.f, 0.f, 0.f};                      // TOK: this pixel's four token logits
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          float x = P1 ? __uint_as_float(v[c]) : fmaf(__uint_as_float(u[c]), 1.0f / 2048.0f, __uint_as_float(v[c]));
          if (EPI == EPI_TOK) {                                  // squeeze: no bias, ReLU; logits from the ReLU-ed value
            x = fmaxf(x, 0.f);
            const float4 wt = *reinterpret_cast<const float4*>(wtok_s + c * 4);
            tl[0] = fmaf(x, wt.x, tl[0]); tl[1] = fmaf(x, wt.y, tl[1]); tl[2] = fmaf(x, wt.z, tl[2]); tl[3] = fmaf(x, wt.w, tl[3]);
          }
          v[c] = __float_as_uint(x);
        }
#pragma unroll
        for (int k4 = 0; k4 < 8; ++k4)
          *reinterpret_cast<float4*>(stage + lane * 32 + ((k4 ^ (lane & 7)) << 2)) =
              make_float4(__uint_as_float(v[k4 * 4]), __uint_as_float(v[k4 * 4 + 1]), __uint_as_float(v[k4 * 4 + 2]), __uint_as_float(v[k4 * 4 + 3]));
        __syncwarp();
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const int r = g * 8 + r4;
          float4 o0 = *reinterpret_cast<const float4*>(stage + r * 32 + (((2 * c4) ^ (r & 7)) << 2));
          float4 o1 = *reinterpret_cast<const float4*>(stage + r * 32 + (((2 * c4 + 1) ^ (r & 7)) << 2));
          o0.x += bia0.x; o0.y += bia0.y; o0.z += bia0.z; o0.w += bia0.w;
          o1.x += bia1.x; o1.y += bia1.y; o1.z += bia1.z; o1.w += bia1.w;
          if (e.res) {
            float4 x0, x1;
            if (e.res_split) { if (P1) half8(ra[g], x0, x1); else join8(ra[g], rb[g], x0, x1); }
            else { x0 = as_f4(ra[g]); x1 = as_f4(rb[g]); }
            o0.x += x0.x; o0.y += x0.y; o0.z += x0.z; o0.w += x0.w;
            o1.x += x1.x; o1.y += x1.y; o1.z += x1.z; o1.w += x1.w;
          }
          if (e.relu) {
            o0.x = fmaxf(o0.x, 0.f); o0.y = fmaxf(o0.y, 0.f); o0.z = fmaxf(o0.z, 0.f); o0.w = fmaxf(o0.w, 0.f);
            o1.x = fmaxf(o1.x, 0.f); o1.y = fmaxf(o1.y, 0.f); o1.z = fmaxf(o1.z, 0.f); o1.w = fmaxf(o1.w, 0.f);
          }
          if (ok[g]) {
            if (P1 && e.out_split) {                             // one FP16 plane (pixel-shuffle as below)
              uint16_t* o16 = reinterpret_cast<uint16_t*>(e.out);
              const size_t off = rowoff[g] + (e.ps ? ((size_t)(j >> 1) * (2 * e.OW) + (j & 1)) * 32 : (size_t)j * 32);
              *reinterpret_cast<uint4*>(o16 + off) = make_uint4(pack_f16x2_sat(o0.x, o0.y), pack_f16x2_sat(o0.z, o0.w),
                                                                pack_f16x2_sat(o1.x, o1.y), pack_f16x2_sat(o1.z, o1.w));
            } else if (!P1 && (EPI == EPI_SPLIT || (EPI == EPI_TOK && e.out_split))) {
              uint4 h, l;
              split8(o0, o1, h, l);
              uint16_t* o16 = reinterpret_cast<uint16_t*>(e.out);
              const size_t off = rowoff[g] + (size_t)j * 32;
              *reinterpret_cast<uint4*>(o16 + off) = h;
              *reinterpret_cast<uint4*>(o16 + off + (size_t)e.out_plane) = l;
            } else {
              // pixel-shuffle store: slab j = (dy, dx) lands on output pixel (2oy + dy, 2ox + dx), 32 channels each
              float* ob = reinterpret_cast<float*>(e.out);
              float* op = e.ps ? ob + rowoff[g] + ((size_t)(j >> 1) * (2 * e.OW) + (j & 1)) * 32 : ob + rowoff[g] + (size_t)j * 32;
              st4(op, o0); st4(op + 4, o1);
            }
          }
        }
        if (e.res && j + 1 < NSLAB) load_res(j + 1);            // next slab's residual: in flight under its TMEM loads
        if (EPI == EPI_TOK) {
          // per-warp online-softmax partials over this warp's 32 pixels (rows still in `stage`), then merged per tile:
          //   m_l = max_p a_pl ; s_l = sum_p exp(a_pl - m_l) ; t_l[c] = sum_p exp(a_pl - m_l) xs_p[c]
          const int mm = q * 32 + lane;
          const bool valid = (t.oy0 + mm / T3_TW < e.OH) && (t.ox0 + mm % T3_TW < e.OW) && (t.n < e.N);
          float ew[4];
#pragma unroll
          for (int l = 0; l < 4; ++l) {
            const float a = valid ? tl[l] : -INFINITY;
            const float mx = warp_max(a);
            ew[l] = valid ? expf(a - mx) : 0.f;
            const float sw = warp_sum(ew[l]);
            if (lane == 0) { tokred[(q * 4 + l) * 34] = mx; tokred[(q * 4 + l) * 34 + 1] = sw; }
          }
          // lane = channel: t_l[c] = sum over the 32 rows; e of row r is fetched with a shuffle
          float ts[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8
          for (int r = 0; r < 32; ++r) {
            const float xv = stage[r * 32 + ((((lane >> 2) ^ (r & 7)) << 2) | (lane & 3))];
#pragma unroll
            for (int l = 0; l < 4; ++l) ts[l] = fmaf(__shfl_sync(0xffffffffu, ew[l], r), xv, ts[l]);
          }
#pragma unroll
          for (int l = 0; l < 4; ++l) tokred[(q * 4 + l) * 34 + 2 + lane] = ts[l];
          asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");   // the four warps of this epilogue group
          // warp q merges token l = q across the four warps and writes the tile's partial
          {
            const int l = q;
            float m4[4], M = -INFINITY;
#pragma unroll
            for (int w4 = 0; w4 < 4; ++w4) { m4[w4] = tokred[(w4 * 4 + l) * 34]; M = fmaxf(M, m4[w4]); }
            float S = 0.f, T = 0.f;
#pragma unroll
            for (int w4 = 0; w4 < 4; ++w4) {
              const float sc = (m4[w4] == -INFINITY) ? 0.f : expf(m4[w4] - M);
              S = fmaf(tokred[(w4 * 4 + l) * 34 + 1], sc, S);
              T = fmaf(tokred[(w4 * 4 + l) * 34 + 2 + lane], sc, T);
            }
            const int mtile = CG == 2 ? 2 * (tile / e.ncout_tiles) + rank : tile / e.ncout_tiles;
            float* pp = e.partials + (((size_t)t.n * e.tiles_per_img + mtile % e.tiles_per_img) * 4 + l) * 34;
            if (t.n < e.N) {
              if (lane == 0) { pp[0] = M; pp[1] = S; }
              pp[2 + lane] = T;
            }
          }
          asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");   // tokred is free for the next tile
        }
        __syncwarp();                                            // the staging rows are free for the next slab
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CG == 2) cluster_sync_all();                      // the peer's shared memory / barriers stay alive until both are done
  if (warp == 1) {
    tc_fence_after();
    if (CG == 2) tmem_dealloc_2sm(tmem_base, Cfg::TMEM_COLS);
    else         tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn3)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn3 get_encode3() {
  static EncodeTiledFn3 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn3)p;
  });
  return fn;
}
struct Key3 {
  const void* ptr; long long d[5];
  bool operator==(const Key3& o) const { return ptr == o.ptr && d[0] == o.d[0] && d[1] == o.d[1] && d[2] == o.d[2] && d[3] == o.d[3] && d[4] == o.d[4]; }
};
struct Key3Hash {
  size_t operator()(const Key3& k) const {
    size_t h = (size_t)k.ptr;
    for (long long v : k.d) h = h * 1000003u ^ (size_t)v;
    return h;
  }
};
std::mutex g_mu3;
std::unordered_map<Key3, CUtensorMap, Key3Hash> g_maps3;

// FP16 activation plane [N][H][W][C] read in {32 ch, bw, bh, 1} boxes (es = element stride along W and H), SWIZZLE_64B
int act_map(CUtensorMap* out, const void* ptr, int C, int W, int H, int N, int bw, int bh, int es) {
  Key3 key{ptr, {C, W, H, ((long long)N << 8) | es, ((long long)bw << 16) | bh}};
  {
    std::lock_guard<std::mutex> lk(g_mu3);
    auto it = g_maps3.find(key);
    if (it != g_maps3.end()) { *out = it->second; return 0; }
  }
  EncodeTiledFn3 enc = get_encode3();
  if (!enc) return DH_E_VARIANT;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)C * W * 2, (cuuint64_t)C * W * H * 2};
  cuuint32_t box[4] = {32, (cuuint32_t)(bw * es), (cuuint32_t)(bh * es), 1};
  cuuint32_t estr[4] = {1, (cuuint32_t)es, (cuuint32_t)es, 1};
  CUtensorMap m;
  const CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return DH_E_SHAPE;
  {
    std::lock_guard<std::mutex> lk(g_mu3);
    if (g_maps3.size() > 4096) g_maps3.clear();
    g_maps3[key] = m;
  }
  *out = m;
  return 0;
}
// filter planes h_w / l_w: [2][Cout][K] FP16 with `plane_bytes` between the planes, read in {32 k, NT rows, `planes`} boxes
// (planes = 2: [h_w ; l_w], 1: h_w alone)
int filt_map(CUtensorMap* out, const void* ptr, int K, int Cout, long long plane_bytes, int NT, int planes) {
  Key3 key{ptr, {K, Cout, plane_bytes, NT, -1 - planes}};
  {
    std::lock_guard<std::mutex> lk(g_mu3);
    auto it = g_maps3.find(key);
    if (it != g_maps3.end()) { *out = it->second; return 0; }
  }
  EncodeTiledFn3 enc = get_encode3();
  if (!enc) return DH_E_VARIANT;
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)Cout, (cuuint64_t)planes};
  cuuint64_t strides[2] = {(cuuint64_t)K * 2, (cuuint64_t)plane_bytes};
  cuuint32_t box[3] = {32, (cuuint32_t)NT, (cuuint32_t)planes};
  cuuint32_t estr[3] = {1, 1, 1};
  CUtensorMap m;
  const CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return DH_E_SHAPE;
  {
    std::lock_guard<std::mutex> lk(g_mu3);
    g_maps3[key] = m;
  }
  *out = m;
  return 0;
}

constexpr uint32_t T3_SMEM_MAX = 232448 - 1024;         // 227 KB opt-in limit minus the static shared memory (barriers)

template <int NT, int KS, int SD, int EPI, bool RES, int CG, bool P1>
int launch3k(const CUtensorMap* A, const CUtensorMap& Bm, const T3Args& e, uint32_t smem, dim3 grid, cudaStream_t s) {
  using Cfg = T3Cfg<NT, RES, CG, P1>;
  auto kern = conv_tc3_kernel<NT, KS, SD, EPI, RES, CG, P1>;
  cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T3_SMEM_MAX);
  if (err != cudaSuccess) return (int)err;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = dim3(Cfg::THREADS, 1, 1); cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[2];
  int na = dh_pdl_attr(at);
  if (CG == 2) {
    at[na].id = cudaLaunchAttributeClusterDimension;
    at[na].val.clusterDim.x = 2; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
    ++na;
  }
  cfg.attrs = at; cfg.numAttrs = na;
  err = cudaLaunchKernelEx(&cfg, kern, A[0], A[1], A[2], A[3], Bm, e);
  if (err != cudaSuccess) return (int)err;
  DH_CHECK_LAUNCH();
  return 0;
}
// the instantiations the network uses: tok = 1x1 / NT 32 / single CTA; everything else by (NT, K, stride, output format).
// P1: one instantiation per geometry, the output format (one FP16 plane or fp32) is read at run time (T3Args::out_split)
template <int NT, bool RES, int CG, bool P1>
int launch3(const CUtensorMap* A, const CUtensorMap& Bm, const T3Args& e, int ks, int stride, int epi, uint32_t smem, dim3 grid, cudaStream_t s) {
  if (epi == EPI_TOK) {
    if constexpr (NT == 32 && CG == 1) return launch3k<32, 1, 1, EPI_TOK, RES, 1, P1>(A, Bm, e, smem, grid, s);
    return DH_E_SHAPE;
  }
  if constexpr (P1) {
    if (stride == 2) return ks == 3 ? launch3k<NT, 3, 2, EPI_SPLIT, RES, CG, true>(A, Bm, e, smem, grid, s) : launch3k<NT, 1, 2, EPI_SPLIT, RES, CG, true>(A, Bm, e, smem, grid, s);
    return ks == 3 ? launch3k<NT, 3, 1, EPI_SPLIT, RES, CG, true>(A, Bm, e, smem, grid, s) : launch3k<NT, 1, 1, EPI_SPLIT, RES, CG, true>(A, Bm, e, smem, grid, s);
  } else {
    if (stride == 2) {
      if (epi == EPI_SPLIT) return ks == 3 ? launch3k<NT, 3, 2, EPI_SPLIT, RES, CG, false>(A, Bm, e, smem, grid, s) : launch3k<NT, 1, 2, EPI_SPLIT, RES, CG, false>(A, Bm, e, smem, grid, s);
      return ks == 3 ? launch3k<NT, 3, 2, EPI_F32, RES, CG, false>(A, Bm, e, smem, grid, s) : launch3k<NT, 1, 2, EPI_F32, RES, CG, false>(A, Bm, e, smem, grid, s);
    }
    if (epi == EPI_SPLIT) return ks == 3 ? launch3k<NT, 3, 1, EPI_SPLIT, RES, CG, false>(A, Bm, e, smem, grid, s) : launch3k<NT, 1, 1, EPI_SPLIT, RES, CG, false>(A, Bm, e, smem, grid, s);
    return ks == 3 ? launch3k<NT, 3, 1, EPI_F32, RES, CG, false>(A, Bm, e, smem, grid, s) : launch3k<NT, 1, 1, EPI_F32, RES, CG, false>(A, Bm, e, smem, grid, s);
  }
}
template <bool RES, int CG, bool P1>
int launch3n(int NT, const CUtensorMap* A, const CUtensorMap& Bm, const T3Args& e, int ks, int stride, int epi, uint32_t smem, dim3 grid, cudaStream_t s) {
  switch (NT) {
    case 128: return launch3<128, RES, CG, P1>(A, Bm, e, ks, stride, epi, smem, grid, s);
    case 64: return launch3<64, RES, CG, P1>(A, Bm, e, ks, stride, epi, smem, grid, s);
    default: return launch3<32, RES, CG, P1>(A, Bm, e, ks, stride, epi, smem, grid, s);
  }
}
template <bool RES>
int launch3c(int cg, bool p1, int NT, const CUtensorMap* A, const CUtensorMap& Bm, const T3Args& e, int ks, int stride, int epi, uint32_t smem,
             dim3 grid, cudaStream_t s) {
  if (p1) return launch3n<RES, 1, true>(NT, A, Bm, e, ks, stride, epi, smem, grid, s);        // no CTA pairs in the single-plane form
  return cg == 2 ? launch3n<RES, 2, false>(NT, A, Bm, e, ks, stride, epi, smem, grid, s)
                 : launch3n<RES, 1, false>(NT, A, Bm, e, ks, stride, epi, smem, grid, s);
}
}  // namespace

bool dh_conv_tc3_eligible(const Conv3Args& a) {
  const bool base = a.in0 && a.wt16 && a.out && (a.stride == 1 || (a.stride == 2 && a.inH % 2 == 0 && a.inW % 2 == 0 && !a.ps)) &&
                    (a.K == 1 || a.K == 3) && a.C0 > 0 && a.C0 % 32 == 0 && a.C1 % 32 == 0 && (a.C1 == 0 || a.in1) &&
                    (a.Cout == 32 || a.Cout == 64 || a.Cout == 128 || a.Cout == 256) && a.inH >= 1 && a.inW >= 1 && a.N >= 1;
  if (!base) return false;
  if (a.ps) return a.Cout == 128 && a.res == nullptr && (!a.out_split || a.h16) && a.K == 3;
  if (a.tok) return a.Cout == 32 && a.K == 1 && a.stride == 1 && a.wtok && a.partials && !a.res && !a.bias;
  return true;
}

int dh_conv_tc3_tok_chunks(int H, int W) { return dh_cdiv(H, T3_TH) * dh_cdiv(W, T3_TW); }

int dh_launch_conv_tc3(const Conv3Args& a, cudaStream_t s) {
  DH_REQUIRE(dh_conv_tc3_eligible(a), DH_E_SHAPE);
  DH_REQUIRE(dh_aligned16(a.in0) && dh_aligned16(a.in1) && dh_aligned16(a.wt16) && dh_aligned16(a.out) &&
             dh_aligned16(a.bias) && dh_aligned16(a.res) && dh_aligned16(a.wtok), DH_E_ALIGN);
  const int Cin = a.C0 + a.C1, K = a.K * a.K * Cin;
  int sms_ = 148, dev_ = 0;
  cudaGetDevice(&dev_);
  cudaDeviceGetAttribute(&sms_, cudaDevAttrMultiProcessorCount, dev_);
  // N tile: 128 output channels — unless that leaves SMs without a tile (small batches: layer3 at 8 pairs has 64 tiles of
  // 128 channels, each a serial chain of 72 (tap, chunk) steps): then 64-channel tiles spread the same work over twice the CTAs
  int NT = a.Cout >= 128 ? 128 : a.Cout;
  if (NT == 128 && !a.ps) {
    const int mt = dh_cdiv(a.inW / a.stride, T3_TW) * dh_cdiv(a.inH / a.stride, T3_TH) * a.N;
    if (mt * (a.Cout / 128) < sms_) NT = 64;
  }
  const int hw = (a.K == 3) ? T3_HW : T3_TW, hh = (a.K == 3) ? T3_HH : T3_TH;
  CUtensorMap A[4], Bm;
  const size_t plane0 = a.in0_plane ? (size_t)a.in0_plane : (size_t)a.N * a.inH * a.inW * a.C0;
  const size_t plane1 = a.in1_plane ? (size_t)a.in1_plane : (size_t)a.N * a.inH * a.inW * a.C1;
  int rc = act_map(&A[0], a.in0, a.C0, a.inW, a.inH, a.N, hw, hh, a.stride);
  if (rc) return rc;
  A[1] = A[0];                                                               // h16: no lo planes
  if (!a.h16) rc = act_map(&A[1], reinterpret_cast<const uint16_t*>(a.in0) + plane0, a.C0, a.inW, a.inH, a.N, hw, hh, a.stride);
  if (rc) return rc;
  if (a.C1) {
    rc = act_map(&A[2], a.in1, a.C1, a.inW, a.inH, a.N, hw, hh, a.stride);
    A[3] = A[2];
    if (!rc && !a.h16) rc = act_map(&A[3], reinterpret_cast<const uint16_t*>(a.in1) + plane1, a.C1, a.inW, a.inH, a.N, hw, hh, a.stride);
    if (rc) return rc;
  } else { A[2] = A[0]; A[3] = A[1]; }
  // CTA pairs: DAHITRA_TC3_CG = 0 (default) never — measured 15-50 % slower on every layer of this network, see DESIGN.md — | 1 on the N = 128 tiles and the K = 1152 -> 32 head conv | 2 always
  static const int env_cg = [] { const char* v = getenv("DAHITRA_TC3_CG"); return v ? atoi(v) : 0; }();
  static const bool env_stream = [] { const char* v = getenv("DAHITRA_TC3_STREAM"); return v && v[0] == '1'; }();   // A/B switch
  const int mtiles = dh_cdiv(a.inW / a.stride, T3_TW) * dh_cdiv(a.inH / a.stride, T3_TH) * a.N;
  int cg = a.tok ? 1 : (a.cg ? a.cg : (env_cg == 2 ? 2 : (env_cg == 1 && (NT == 128 || (a.Cout == 32 && K >= 1152)) ? 2 : 1)));
  DH_REQUIRE(!(a.h16 && cg == 2), DH_E_VARIANT);                           // the single-plane form has no CTA-pair variant
  if (mtiles < 2) cg = 1;
  rc = filt_map(&Bm, a.wt16, K, a.Cout, a.wt_plane_bytes, NT / cg, a.h16 ? 1 : 2);
  if (rc) return rc;
  T3Args e;
  e.bias = a.bias; e.res = a.res; e.out = a.out; e.wtok = a.wtok; e.partials = a.partials;
  e.OH = a.inH / a.stride; e.OW = a.inW / a.stride; e.Cout = a.Cout; e.relu = a.relu;
  e.tilesX = dh_cdiv(e.OW, T3_TW); e.tilesY = dh_cdiv(e.OH, T3_TH);
  e.cchunks0 = a.C0 / 32; e.cchunks = Cin / 32; e.Cin = Cin; e.ps = a.ps; e.N = a.N;
  e.ncout_tiles = a.Cout / NT;
  e.tiles_per_img = e.tilesX * e.tilesY;
  e.ntiles = (cg == 2 ? (mtiles + 1) / 2 : mtiles) * e.ncout_tiles;        // work items: tiles, or tile pairs
  e.res_split = a.res_split; e.out_split = a.out_split;
  e.res_plane = a.res_plane ? a.res_plane : (long long)a.N * e.OH * e.OW * a.Cout;
  e.out_plane = a.out_plane ? a.out_plane : (long long)a.N * e.OH * e.OW * a.Cout;
  e.halo_plane_bytes = (uint32_t)(hw * hh * 64);
  const int epi = a.tok ? EPI_TOK : ((a.out_split || a.h16) ? EPI_SPLIT : EPI_F32);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int slots = sms / cg;                                                // persistent: one CTA (pair) per SM (TPC)
  const int nwork = e.ntiles < slots ? e.ntiles : slots;
  dim3 grid((unsigned)(nwork * cg), 1, 1);
  // resident filter when the whole [h_w ; l_w] image (h16: h_w; a CTA of a pair: its half) fits next to two halo buffers, and
  // every CTA walks enough tiles to amortise loading it (otherwise the streaming ring, whose first MMA starts after one stage)
  const uint32_t w_bytes = (uint32_t)K * (uint32_t)a.Cout * (a.h16 ? 2u : 4u) / (uint32_t)cg;   // = ncout_tiles * cchunks * taps * B_TAP
  const uint32_t halo = a.h16 ? T3_PLANE : T3_HALO;                        // one halo buffer
  const uint32_t fixed = 8 * 4096 + 1024 + (a.tok ? 512 + 2 * 2176 : 0);   // epilogue staging (8 warps) + alignment slack (+ tok scratch)
  const bool res_ok = w_bytes + 2 * halo + fixed <= T3_SMEM_MAX && !a.force_stream && !env_stream && e.ntiles >= 2 * nwork;
  if (res_ok) {
    int hb = (int)((T3_SMEM_MAX - fixed - w_bytes) / halo);
    e.hb = hb > T3_MAX_HB ? T3_MAX_HB : hb;
    const uint32_t smem = (uint32_t)e.hb * halo + w_bytes + fixed;
    return launch3c<true>(cg, a.h16, NT, A, Bm, e, a.K, a.stride, epi, smem, grid, s);
  }
  e.hb = T3_MAX_HB;
  const uint32_t ring = a.h16 ? (NT == 128 ? T3Cfg<128, false, 1, true>::RING_BYTES : (NT == 64 ? T3Cfg<64, false, 1, true>::RING_BYTES : T3Cfg<32, false, 1, true>::RING_BYTES))
                              : (NT == 128 ? T3Cfg<128, false>::RING_BYTES : (NT == 64 ? T3Cfg<64, false>::RING_BYTES : T3Cfg<32, false>::RING_BYTES));
  const uint32_t smem = T3_MAX_HB * halo + ring + fixed;                  // the pair's ring has twice the stages of half the size
  return launch3c<false>(cg, a.h16, NT, A, Bm, e, a.K, a.stride, epi, smem, grid, s);
}
