// dahitra_b200 — implicit-GEMM convolution on tcgen05, halo-reuse variant (stride 1, 3x3 or 1x1), with an
// optional error-compensated 3xTF32 mode that brings the tensor-core path to fp32-grade accuracy.
//
//   D[m][co] = sum_{chunk, tap, ci} X[pixel(m) + tap][chunk*32 + ci] * Wt[co][tap*Cin + chunk*32 + ci]
//   M tile = 128 output pixels = 16 rows x 8 columns of one image  (row m = y*8 + x: every 8-row UMMA atom is
//            8 horizontally adjacent pixels)
//   For each 32-channel chunk the (16+2) x (8+2) input HALO is fetched ONCE by one 4-D TMA box {32ch,10,18,1}
//   (zero-filled outside the image = the conv padding) and stays in shared memory for all 9 taps: the A operand
//   of tap (r,s) is the SAME buffer addressed through a UMMA descriptor whose start is shifted by (r*10+s) pixels
//   (x128 B) with a stride-byte-offset of 10 pixels.  tcgen05 applies the 128B-swizzle XOR on absolute
//   shared-memory address bits, so a row-shifted window of a TMA-written tile is read back correctly
//   (measured: tools/umma_probe.cu).  L2->SM activation traffic drops 9x -> 1.4x versus conv_tc.cu.
//   The filter tile of each (chunk, tap) streams through a TMA ring (K-major [Cout][K], box {32, NT}).
//
// 3xTF32 (X3): activations are split in shared memory by four extra warps, once per halo chunk
// (hi = cvt.rna.tf32(v) in place, lo = v - hi into a twin buffer); filters arrive pre-split (hi / lo arrays);
// each K step issues A_hi.B_hi + A_lo.B_hi + A_hi.B_lo.  The split costs one smem pass per chunk, amortised
// over 9 taps.
//
// XM = 2 ("3xTF32 with bf16 corrections"): the two correction products A_lo.B_hi and A_hi.B_lo only have to be right to
// ~8 bits (they are 2^-11 of the main term), so they run as kind::f16 BF16 MMAs — K = 16 per instruction, i.e. half the
// MMAs and half the operand bytes of their TF32 form.  The splitter then writes, next to the TF32-rounded fp32 halo, two
// bf16 halos (bf16(a) and bf16(a - tf32(a)), 64-byte pixel rows in the SWIZZLE_64B pattern — the shifted-window trick
// works there too, tools/umma_bf16_probe.cu), and the filter ring carries bf16(w) and bf16(w - tf32(w)) tiles.
// Per (tap, 32-channel chunk): 4 TF32 + 2 + 2 BF16 MMAs instead of 12.
//
// XM = 4: like XM = 2 with the MAIN product in FP16 (11-bit significand like TF32, but 16-bit operands: K = 16 per MMA,
// half the operand bytes): a = f16(a) + r_a, w = f16(w) + r_w with the remainders carried in bf16 (fp32 range, so values
// beyond the f16 range — saturated to +-65504 — or below its normal range only cost accuracy of the correction terms).
// Per (tap, chunk): 2 FP16 + 2 + 2 BF16 MMAs.  The splitter writes three 16-bit halos: f16(a), bf16(a), bf16(a - f16(a)).
//
// XM = 6: XM = 4 with the third product folded into the first.  a.w = f16(a).f16(w) + r_a.bf16(w) + f16(a).r_w: the first
// and third products share the A operand, so the filter tile is the 2N-row concatenation [f16(w) ; f16(2^11 r_w)] and ONE
// N-doubled FP16 MMA produces both (the scaled remainder keeps r_w in the normal FP16 range); they land in two column
// blocks of the accumulator and the epilogue adds them (main + 2^-11 corr).  Per (tap, chunk): 2 wide + 2 narrow MMAs
// instead of 6 — a third fewer A-operand reads, which is what bounds the N = 32 / 64 tiles.  Two 16-bit halos only.
//
// XM = 3 ("bf16"): single-pass BF16 operands (fp32 storage, fp32 accumulation): the splitter only converts the halo to
// the bf16 tile, the ring only carries bf16(w); 2 MMAs per (tap, chunk).  Separately stated tolerance (tests).
//
// Stride 2 (SD = 2; resnet layer2.0): the input is read as its four 2x2 phase images P_ab(y,x) = X(2y+a, 2x+b),
// each fetched by a TMA box with elementStrides {1,2,2,1}.  A 3x3 stride-2 tap (r,s) is the stride-1 tap of phase
// (r odd ? 0 : 1, s odd ? 0 : 1) at offset (r == 0 ? -1 : 0, s == 0 ? -1 : 0), so every (chunk, phase) pair is one
// 18x10 halo serving 1, 2, 2 or 4 taps through the same shifted-window descriptors.
//
// Persistent CTAs (one per SM) walk the tile list; two TMEM accumulators let the epilogue of tile i overlap the
// main loop of tile i+1.  Warp roles: 0 = halo TMA producer, 1 = TMEM alloc + MMA issuer, 2..5 = epilogue,
// 6 = filter TMA producer, 7..10 = splitter (X3 only).
#include "tc_common.cuh"
#include <mutex>
#include <unordered_map>

using namespace dhtc;

namespace {

constexpr int T2_TH = 16, T2_TW = 8;                    // output patch
constexpr int T2_HW = T2_TW + 2, T2_HH = T2_TH + 2;     // halo 10 x 18
constexpr uint32_t T2_HALO_STRIDE = 23552;              // 1024-aligned
constexpr uint32_t T2_HALO16_BYTES = T2_HW * T2_HH * 64; // one bf16 halo (11520 B); two of them share a "lo" buffer

struct T2Args {
  const float* bias; const float* res; float* out;
  int OH, OW, Cout, relu, tilesX, cchunks0, cchunks, ntaps, KW, Cin, ps;
  int halo_w, halo_h;        // 10 x 18 (3x3) or 8 x 16 (1x1)
  int stride;                // 1 or 2
  int tilesY, ncout_tiles, ntiles;   // ntiles: work items = tiles (CG = 1) or tile pairs (CG = 2)
  int N;                             // images
  uint32_t halo_bytes;
};

template <int NT, int XM, int CG = 1> struct T2Cfg {
  static constexpr bool X3 = XM != 0;              // modes with a splitter pass: 1 = three TF32 MMAs, 2 = TF32 + two BF16, 3 = BF16 only
  // Persistent kernel, one CTA per SM.  Pipeline depth is sized so that the MMA warp always has >= ~1500 cycles of
  // operands in flight (L2 latency under load): the smaller the N tile, the faster a stage is consumed, so the more
  // halo buffers (HB) and filter stages it gets.  A stage holds TPS filter taps so the issuing thread waits /
  // commits once per 4*TPS (x3: 12*TPS) MMAs.
  static constexpr int HB = X3 ? 2 : (NT == 128 ? 2 : (NT == 64 ? 3 : 4));          // halo chunk buffers (x3: hi + lo each)
  static constexpr bool ONE16 = (XM == 3 || XM == 5);   // single-pass 16-bit operands: 3 = bf16, 5 = f16 (saturating)
  static constexpr int TPS = ONE16 ? 3 : (X3 ? (NT == 32 ? 3 : 1) : 3);
  static constexpr int STAGES1 = ONE16 ? (NT == 128 ? 4 : (NT == 64 ? 6 : 8))
                               : (X3 ? (NT == 128 ? 3 : (NT == 64 ? 6 : 4)) : (NT == 128 ? 3 : (NT == 64 ? 5 : 8)));
  static constexpr int STAGES = CG == 2 ? (2 * STAGES1 > 8 ? 8 : 2 * STAGES1) : STAGES1;   // CTA pair: half-size B tiles
  static constexpr uint32_t B_TILE = (NT / CG) * 128;           // a CTA of a pair holds N/2 rows of B
  static constexpr bool WIDE = XM == 6;             // accumulator = [main + corr2 | 2^11 corr3]: 2 NT columns
  static constexpr uint32_t B_TAP = ONE16 ? B_TILE / 2 : ((XM == 4 || XM == 6) ? 3 * (B_TILE / 2) : B_TILE * (X3 ? 2 : 1));
  // XM 0: fp32 | 1: fp32 hi, lo | 2: fp32 hi, bf16 hi, lo | 3: bf16 | 4: f16, bf16 hi, bf16 lo
  static constexpr uint32_t LO_STRIDE = XM == 4 ? 35840u : 23552u;   // the 16-bit halos of one buffer (XM = 4: three of 11520 B)
  static constexpr uint32_t IDESCF = umma_idesc_f16(128 * CG, NT);
  static constexpr uint32_t IDESCF_WIDE = umma_idesc_f16(128 * CG, 2 * NT);
  static constexpr int ACC_COLS = WIDE ? 2 * NT : NT;                       // TMEM columns of one accumulator
  static constexpr uint32_t IDESC16 = umma_idesc_bf16(128 * CG, NT);
  static constexpr uint32_t B_STAGE = B_TAP * TPS;
  static constexpr uint32_t HALO_BYTES = HB * T2_HALO_STRIDE + (X3 ? HB * LO_STRIDE : 0);   // [hi 0..HB-1][lo 0..HB-1]
  static constexpr uint32_t EPI_OFF = HALO_BYTES + STAGES * B_STAGE;   // epilogue staging: 4 warps x 4 KB
  static constexpr uint32_t SMEM = EPI_OFF + 4 * 4096 + 1024;
  static constexpr int THREADS = X3 ? 352 : 224;                // + 4 splitter warps
  static constexpr uint32_t IDESC = umma_idesc_tf32(128 * CG, NT);
  static constexpr uint32_t TMEM_COLS = (2 * ACC_COLS < 32) ? 32 : 2 * ACC_COLS;   // two accumulators
};

__device__ __forceinline__ float tf32_rna(float v) { return tf32_round(v); }

// shifted-window A descriptor: start = halo + (r*halo_w + s) pixels, SBO = halo_w pixels
__device__ __forceinline__ uint64_t halo_desc(uint32_t addr, uint32_t sbo_bytes) {
  return (uint64_t)((addr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}

// Order in which the nine 3x3 taps are consumed and the halo-pixel shift of each.
//   stride 1: one halo per chunk, taps 0..8, shift (r, s)
//   stride 2: four halos per chunk (phase = 2a + b), taps grouped by phase, shift (r != 0, s != 0)
template <int KS, int SD> struct TapSched {
  static constexpr int NPH = (KS == 3 && SD == 2) ? 4 : 1;
  static constexpr int NTAPS = KS * KS;
  __host__ __device__ static constexpr int tap(int i) {
    return (KS == 3 && SD == 2) ? (int)((0x862071534ULL >> (4 * i)) & 0xF) : i;   // {4, 3,5, 1,7, 0,2,6,8}, nibble-packed
  }
  __host__ __device__ static constexpr int first(int ph) {           // index of the first tap of phase ph (first(NPH) = NTAPS)
    return (KS == 3 && SD == 2) ? (int)((0x95310u >> (4 * ph)) & 0xF) : (ph == 0 ? 0 : NTAPS);   // {0, 1, 3, 5, 9}
  }
  __host__ __device__ static constexpr int shift_px(int t, int halo_w) {
    return KS == 1 ? 0 : (SD == 2 ? ((t / 3 != 0) ? halo_w : 0) + ((t % 3 != 0) ? 1 : 0) : (t / 3) * halo_w + t % 3);
  }
};

struct TileCoord { int n, oy0, ox0, n0; };
// CG = 2: work item = (pair of consecutive M tiles, cout tile); CTA `rank` of the pair takes M tile 2*pair + rank.  The
// odd tile of the last pair may not exist: then n == e.N, its TMA boxes are out of bounds (zero-filled) and its
// epilogue stores nothing.
__device__ __forceinline__ TileCoord tile_coord(int tile, const T2Args& e, int NT, int CG = 1, int rank = 0) {
  TileCoord t;
  const int ct = tile % e.ncout_tiles; tile /= e.ncout_tiles;
  if (CG == 2) tile = 2 * tile + rank;
  const int tx = tile % e.tilesX; tile /= e.tilesX;
  const int ty = tile % e.tilesY;
  t.n = tile / e.tilesY; t.oy0 = ty * T2_TH; t.ox0 = tx * T2_TW; t.n0 = ct * NT;
  return t;
}

template <int NT, int XM, int KS, int SD, int CG>
__global__ void __launch_bounds__(T2Cfg<NT, XM, CG>::THREADS, 1)
conv_tc2_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
                const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmB16,
                const __grid_constant__ CUtensorMap tmB16f, const T2Args e) {
  using Cfg = T2Cfg<NT, XM, CG>;
  constexpr bool X3 = XM != 0;
  static_assert(XM < 3 || CG == 1, "the 16-bit-main modes are implemented for single-CTA tiles");
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t t2_raw[];
  constexpr int HB = Cfg::HB;
  __shared__ __align__(8) uint64_t halo_full[HB], halo_ready[HB], halo_empty[HB], b_full[STAGES], b_empty[STAGES],
      acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t base = (smem_u32(t2_raw) + 1023u) & ~1023u;
  uint8_t* base_ptr = t2_raw + (base - smem_u32(t2_raw));
  const uint32_t b_ring = base + Cfg::HALO_BYTES;
  constexpr uint32_t LO0 = (uint32_t)Cfg::HB * T2_HALO_STRIDE;          // offset of the first "lo" buffer
  constexpr int pad = (KS == 3) ? 1 : 0;
  using Sched = TapSched<KS, SD>;
  constexpr int NPH = Sched::NPH;
  // CTA pair (CG = 2): rank 0 is the leader — it alone issues the MMAs and owns the barriers the MMA warp waits on
  // (halo_ready / halo_full in 1xTF32 / b_full / acc_empty); the peer's producers, splitters and epilogue signal them
  // remotely, and the leader's multicast commits release the *_empty / acc_full barriers of both CTAs.
  const int rank = CG == 2 ? (int)cluster_ctarank() : 0;
  const int w0 = CG == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;          // first work item, and the stride between items
  const int wstep = CG == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (threadIdx.x == 0) {
    for (int i = 0; i < HB; ++i) {
      mbar_init(smem_u32(&halo_full[i]), 1);
      mbar_init(smem_u32(&halo_ready[i]), 128 * CG);  // X3: every splitter thread (of both CTAs) arrives
      mbar_init(smem_u32(&halo_empty[i]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&acc_full[i]), 1);
      mbar_init(smem_u32(&acc_empty[i]), 128 * CG);   // every epilogue thread (of both CTAs) arrives
    }
    for (int s = 0; s < STAGES; ++s) { mbar_init(smem_u32(&b_full[s]), 1); mbar_init(smem_u32(&b_empty[s]), 1); }
    mbar_fence_init();
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA0) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
  }
  if (warp == 1) {
    if (CG == 2) tmem_alloc_2sm(smem_u32(&tmem_slot), Cfg::TMEM_COLS);
    else         tmem_alloc(smem_u32(&tmem_slot), Cfg::TMEM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  if (CG == 2) cluster_sync_all();                      // the peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  // Every role walks the same tile sequence tile = blockIdx.x, += gridDim.x and keeps its own running counters:
  //   g  = halo chunks consumed so far (buffer g&1, use number g>>1), step = filter ring stages so far,
  //   it = tiles so far (accumulator it&1, use number it>>1).
  if (warp == 0) {
    if (lane == 0) {                                            // ---------------- halo TMA producer
      int g = 0;
      for (int tile = w0; tile < e.ntiles; tile += wstep) {
        const TileCoord t = tile_coord(tile, e, NT, CG, rank);
        for (int cc = 0; cc < e.cchunks; ++cc) {
#pragma unroll
          for (int ph = 0; ph < NPH; ++ph, ++g) {
            const int hb = g % HB, use = g / HB;
            mbar_wait(smem_u32(&halo_empty[hb]), (uint32_t)((use & 1) ^ 1));
            // 1xTF32 pair: the MMA warp waits on the LEADER's halo_full, which counts the bytes of both halos
            constexpr bool REMOTE = (CG == 2 && !X3);
            const uint32_t bar = smem_u32(&halo_full[hb]);
            if (!REMOTE) mbar_expect_tx(bar, e.halo_bytes);
            else if (rank == 0) mbar_expect_tx(bar, 2 * e.halo_bytes);
            const uint32_t dst = base + (uint32_t)hb * T2_HALO_STRIDE;
            // input coordinates of the halo origin (stride 2: origin of phase (ph>>1, ph&1), in full-resolution pixels)
            const int cx = SD == 1 ? t.ox0 - pad : 2 * (t.ox0 - pad) + (ph & 1);
            const int cy = SD == 1 ? t.oy0 - pad : 2 * (t.oy0 - pad) + (ph >> 1);
            const CUtensorMap* tm = cc < e.cchunks0 ? &tmA0 : &tmA1;
            const int c0 = (cc < e.cchunks0 ? cc : cc - e.cchunks0) * 32;
            if (REMOTE && rank == 1) tma_load_4d_2sm(dst, tm, mapa_u32(bar, 0), c0, cx, cy, t.n);
            else                     tma_load_4d(dst, tm, bar, c0, cx, cy, t.n);
          }
        }
      }
    }
  } else if (warp == 6) {
    if (lane == 0) {                                            // ---------------- filter TMA producer
      constexpr int NTAPS_ = KS * KS;
      constexpr int TPS_ = (SD == 1 && NTAPS_ % Cfg::TPS == 0) ? Cfg::TPS : 1;
      int step = 0;
      for (int tile = w0; tile < e.ntiles; tile += wstep) {
        const TileCoord t = tile_coord(tile, e, NT, CG, rank);
        for (int cc = 0; cc < e.cchunks; ++cc) {
#pragma unroll
          for (int i0 = 0; i0 < NTAPS_; i0 += TPS_, ++step) {              // one ring stage = TPS_ filter taps, in schedule order
            const int st = step % STAGES, round = step / STAGES;
            mbar_wait(smem_u32(&b_empty[st]), (uint32_t)((round & 1) ^ 1));
            const uint32_t bar = smem_u32(&b_full[st]);                    // CG = 2: the leader's barrier counts both halves
            if (rank == 0) mbar_expect_tx(bar, (uint32_t)(CG * TPS_) * Cfg::B_TAP);
            const uint32_t lbar = (CG == 2 && rank == 1) ? mapa_u32(bar, 0) : bar;
            const int nrow = t.n0 + rank * (NT / CG);
#pragma unroll
            for (int tt = 0; tt < TPS_; ++tt) {
              const uint32_t dst = b_ring + (uint32_t)st * Cfg::B_STAGE + (uint32_t)tt * Cfg::B_TAP;
              const int kcol = Sched::tap(i0 + tt) * e.Cin + cc * 32;
              if (CG == 2 && rank == 1) {
                tma_load_2d_2sm(dst, &tmB, lbar, kcol, nrow);
                if (XM == 2) {
                  tma_load_2d_2sm(dst + Cfg::B_TILE, &tmB16, lbar, kcol, nrow);
                  tma_load_2d_2sm(dst + Cfg::B_TILE + Cfg::B_TILE / 2, &tmB16, lbar, kcol, e.Cout + nrow);
                } else if (X3) {
                  tma_load_2d_2sm(dst + Cfg::B_TILE, &tmB, lbar, kcol, e.Cout + nrow);
                }
              } else if (XM == 6) {
                tma_load_2d(dst, &tmB16f, bar, kcol, nrow);                                        // f16(w)            \ one 2N-row
                tma_load_2d(dst + Cfg::B_TILE / 2, &tmB, bar, kcol, nrow);                         // f16(2^11 r_w)     /  B tile   (tmB = plane 4 here)
                tma_load_2d(dst + Cfg::B_TILE, &tmB16, bar, kcol, nrow);                           // bf16(w)
              } else if (XM == 4) {
                tma_load_2d(dst, &tmB16f, bar, kcol, nrow);                                        // f16(w)
                tma_load_2d(dst + Cfg::B_TILE / 2, &tmB16, bar, kcol, nrow);                       // bf16(w)
                tma_load_2d(dst + Cfg::B_TILE, &tmB16f, bar, kcol, e.Cout + nrow);                 // bf16(w - f16(w))
              } else if (XM == 5) {
                tma_load_2d(dst, &tmB16f, bar, kcol, nrow);                                        // f16(w) only
              } else if (XM == 3) {
                tma_load_2d(dst, &tmB16, bar, kcol, nrow);                                         // bf16(w) only
              } else if (XM == 2) {
                tma_load_2d(dst, &tmB, bar, kcol, nrow);                                           // fp32 (TF32-rounded) filter
                tma_load_2d(dst + Cfg::B_TILE, &tmB16, bar, kcol, nrow);                           // bf16(w)
                tma_load_2d(dst + Cfg::B_TILE + Cfg::B_TILE / 2, &tmB16, bar, kcol, e.Cout + nrow); // bf16(w - tf32(w))
              } else {
                tma_load_2d(dst, &tmB, bar, kcol, nrow);
                if (X3) tma_load_2d(dst + Cfg::B_TILE, &tmB, bar, kcol, e.Cout + nrow);  // lo rows follow the hi rows
              }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {                               // ---------------- MMA issuer (pair: the leader only)
      // The issuing thread is the critical path of the whole kernel: everything between two tcgen05.mma's is
      // compile-time (tap shifts, taps per stage) or a wrapping counter — no divisions, no runtime tap arithmetic.
      constexpr int NTAPS = KS * KS;
      constexpr int HALO_W = (KS == 3) ? T2_HW : T2_TW;
      constexpr int TPS = (SD == 1 && NTAPS % Cfg::TPS == 0) ? Cfg::TPS : 1;
      constexpr uint32_t SBO = (uint32_t)HALO_W * 128u;
      auto mma = [](uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
        if (CG == 2) umma_tf32_2sm(d, a, b, idesc, acc); else umma_tf32(d, a, b, idesc, acc);
      };
      auto mma16 = [](uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
        if (CG == 2) umma_bf16_2sm(d, a, b, idesc, acc); else umma_bf16(d, a, b, idesc, acc);
      };
      auto commit = [](uint32_t bar) { if (CG == 2) umma_commit_2sm(bar); else umma_commit(bar); };
      int hb = 0, st = 0;
      uint32_t hphase = 0, bphase = 0;
      int it = 0;
      for (int tile = w0; tile < e.ntiles; tile += wstep, ++it) {
        const int ab = it & 1;
        if (CG == 2) mbar_wait_cluster(smem_u32(&acc_empty[ab]), (uint32_t)(((it >> 1) & 1) ^ 1));
        else         mbar_wait(smem_u32(&acc_empty[ab]), (uint32_t)(((it >> 1) & 1) ^ 1));    // epilogue drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)ab * Cfg::ACC_COLS;
        for (int cc = 0; cc < e.cchunks; ++cc) {
#pragma unroll
          for (int ph = 0; ph < NPH; ++ph) {
            if (X3 && CG == 2) mbar_wait_cluster(smem_u32(&halo_ready[hb]), hphase);
            else if (X3)       mbar_wait(smem_u32(&halo_ready[hb]), hphase);
            else               mbar_wait(smem_u32(&halo_full[hb]), hphase);
            tc_fence_after();
            const uint32_t h_hi = base + (uint32_t)hb * T2_HALO_STRIDE;
            const uint64_t ah0 = halo_desc(h_hi, SBO);
            const uint32_t h_lo = base + LO0 + (uint32_t)hb * Cfg::LO_STRIDE;                     // this buffer's 16-bit halos / fp32 lo
            const uint64_t al0 = halo_desc(h_lo, SBO);
#pragma unroll
            for (int i0 = Sched::first(ph); i0 < Sched::first(ph + 1); i0 += TPS) {
              mbar_wait(smem_u32(&b_full[st]), bphase);
              tc_fence_after();
              const uint32_t b_stage = b_ring + (uint32_t)st * Cfg::B_STAGE;
#pragma unroll
              for (int tt = 0; tt < TPS; ++tt) {
                const int i = i0 + tt;
                const uint32_t shift16 = (uint32_t)(Sched::shift_px(Sched::tap(i), HALO_W) * 128) >> 4;   // compile-time after unrolling
                const uint64_t ah = ah0 + (uint64_t)shift16;
                const uint64_t bh = umma_desc_sw128(b_stage + (uint32_t)tt * Cfg::B_TAP);
                if (XM == 6) {
                  // [f16(a)] x [f16 w ; f16 2^11 r_w] as one 2N-wide MMA, then [bf16 r_a] x [bf16 w] into the first N columns
                  constexpr uint32_t SBO16 = (uint32_t)HALO_W * 64u;
                  const uint32_t px = (uint32_t)Sched::shift_px(Sched::tap(i), HALO_W) * 64u;
                  const uint64_t a_f = umma_desc_sw64(h_lo + px, SBO16), a_r = umma_desc_sw64(h_lo + T2_HALO16_BYTES + px, SBO16);
                  const uint32_t bt = b_stage + (uint32_t)tt * Cfg::B_TAP;
                  const uint64_t b_w = umma_desc_sw64(bt, 512u), b_b = umma_desc_sw64(bt + Cfg::B_TILE, 512u);
#pragma unroll
                  for (int k = 0; k < 2; ++k) mma16(d_tmem, a_f + (uint64_t)(2 * k), b_w + (uint64_t)(2 * k), Cfg::IDESCF_WIDE, (cc | i | k) ? 1u : 0u);
#pragma unroll
                  for (int k = 0; k < 2; ++k) mma16(d_tmem, a_r + (uint64_t)(2 * k), b_b + (uint64_t)(2 * k), Cfg::IDESC16, 1u);
                } else if (XM == 4) {
                  // f16 main product + two bf16 corrections; halos [f16(a)][bf16(a)][bf16(a - f16(a))], filter [f16 w][bf16 w][bf16 r_w]
                  constexpr uint32_t SBO16 = (uint32_t)HALO_W * 64u;
                  const uint32_t px = (uint32_t)Sched::shift_px(Sched::tap(i), HALO_W) * 64u;
                  const uint64_t a_f = umma_desc_sw64(h_lo + px, SBO16), a_b = umma_desc_sw64(h_lo + T2_HALO16_BYTES + px, SBO16),
                                 a_r = umma_desc_sw64(h_lo + 2 * T2_HALO16_BYTES + px, SBO16);
                  const uint32_t bt = b_stage + (uint32_t)tt * Cfg::B_TAP;
                  const uint64_t b_f = umma_desc_sw64(bt, 512u), b_b = umma_desc_sw64(bt + Cfg::B_TILE / 2, 512u),
                                 b_r = umma_desc_sw64(bt + Cfg::B_TILE, 512u);
#pragma unroll
                  for (int k = 0; k < 2; ++k) mma16(d_tmem, a_f + (uint64_t)(2 * k), b_f + (uint64_t)(2 * k), Cfg::IDESCF, (cc | i | k) ? 1u : 0u);
#pragma unroll
                  for (int k = 0; k < 2; ++k) mma16(d_tmem, a_r + (uint64_t)(2 * k), b_b + (uint64_t)(2 * k), Cfg::IDESC16, 1u);
#pragma unroll
                  for (int k = 0; k < 2; ++k) mma16(d_tmem, a_b + (uint64_t)(2 * k), b_r + (uint64_t)(2 * k), Cfg::IDESC16, 1u);
                } else if (XM == 3 || XM == 5) {
                  // single-pass 16-bit operands: A = the bf16 / f16 halo (first tile of the "lo" buffer), B = the matching filter tile
                  const uint32_t h16 = h_lo + (uint32_t)Sched::shift_px(Sched::tap(i), HALO_W) * 64u;
                  const uint64_t a16 = umma_desc_sw64(h16, (uint32_t)HALO_W * 64u);
                  const uint64_t b16 = umma_desc_sw64(b_stage + (uint32_t)tt * Cfg::B_TAP, 512u);
#pragma unroll
                  for (int k = 0; k < 2; ++k)
                    mma16(d_tmem, a16 + (uint64_t)(2 * k), b16 + (uint64_t)(2 * k), XM == 5 ? Cfg::IDESCF : Cfg::IDESC16, (cc | i | k) ? 1u : 0u);
                } else {
#pragma unroll
                  for (int k = 0; k < 4; ++k) mma(d_tmem, ah + (uint64_t)(2 * k), bh + (uint64_t)(2 * k), Cfg::IDESC, (cc | i | k) ? 1u : 0u);
                }
                if (XM == 2) {
                  // corrections in bf16: A = the bf16 halos (64-byte pixel rows), B = the bf16 filter tiles; K = 16 per MMA
                  constexpr uint32_t SBO16 = (uint32_t)HALO_W * 64u;
                  const uint32_t px = (uint32_t)Sched::shift_px(Sched::tap(i), HALO_W) * 64u;
                  const uint32_t h16 = h_lo;                                           // [bf16(a)][bf16(a - tf32(a))]
                  const uint64_t a_hi16 = umma_desc_sw64(h16 + px, SBO16), a_lo16 = umma_desc_sw64(h16 + T2_HALO16_BYTES + px, SBO16);
                  const uint32_t b16 = b_stage + (uint32_t)tt * Cfg::B_TAP + Cfg::B_TILE;
                  const uint64_t b_hi16 = umma_desc_sw64(b16, 512u), b_lo16 = umma_desc_sw64(b16 + Cfg::B_TILE / 2, 512u);
#pragma unroll
                  for (int k = 0; k < 2; ++k) mma16(d_tmem, a_lo16 + (uint64_t)(2 * k), b_hi16 + (uint64_t)(2 * k), Cfg::IDESC16, 1u);
#pragma unroll
                  for (int k = 0; k < 2; ++k) mma16(d_tmem, a_hi16 + (uint64_t)(2 * k), b_lo16 + (uint64_t)(2 * k), Cfg::IDESC16, 1u);
                } else if (XM == 1) {
                  const uint64_t al = al0 + (uint64_t)shift16;
                  const uint64_t bl = umma_desc_sw128(b_stage + (uint32_t)tt * Cfg::B_TAP + Cfg::B_TILE);
#pragma unroll
                  for (int k = 0; k < 4; ++k) mma(d_tmem, al + (uint64_t)(2 * k), bh + (uint64_t)(2 * k), Cfg::IDESC, 1u);
#pragma unroll
                  for (int k = 0; k < 4; ++k) mma(d_tmem, ah + (uint64_t)(2 * k), bl + (uint64_t)(2 * k), Cfg::IDESC, 1u);
                }
              }
              commit(smem_u32(&b_empty[st]));
              if (++st == STAGES) { st = 0; bphase ^= 1u; }
            }
            commit(smem_u32(&halo_empty[hb]));             // all taps of this halo have been issued
            if (++hb == HB) { hb = 0; hphase ^= 1u; }
          }
        }
        commit(smem_u32(&acc_full[ab]));
      }
    }
  } else if (warp < 6) {                                        // ---------------- epilogue (warps 2..5)
    // Each thread owns one accumulator row (pixel), but a store instruction in which every lane writes 16 bytes of a
    // different 128-byte line costs 32 L1 passes — cycles taken from the same data pipe that feeds the MMA operands.
    // So every 32-channel slab goes through a per-warp shared-memory transpose: rows in (8 conflict-free 16-byte
    // stores), then 8 lanes per pixel row out, 4 whole 128-byte lines per instruction for the residual read and the store.
    const int q = warp & 3;
    const int m = q * 32 + lane;
    float* stage = reinterpret_cast<float*>(base_ptr + Cfg::EPI_OFF + (size_t)q * 4096);   // [32 rows][8 chunks ^ (row & 7)][4]
    const int c8 = lane & 7, r8 = lane >> 3;                    // phase 2: lane -> (chunk of 4 channels, row within a group of 4)
    int it = 0;
    for (int tile = w0; tile < e.ntiles; tile += wstep, ++it) {
      const TileCoord t = tile_coord(tile, e, NT, CG, rank);
      const int ab = it & 1;
      mbar_wait(smem_u32(&acc_full[ab]), (uint32_t)((it >> 1) & 1));
      tc_fence_after();
      // phase-2 coordinates of this lane's 8 rows (row r = g*4 + r8 of the warp's 32 = pixel (y = 4q + r/8, x = r%8))
      size_t rowoff[8];
      bool ok[8];
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        const int mm = q * 32 + g * 4 + r8;
        const int oy = t.oy0 + mm / T2_TW, ox = t.ox0 + mm % T2_TW;
        ok[g] = (oy < e.OH) && (ox < e.OW) && (t.n < e.N);
        rowoff[g] = e.ps ? ((size_t)(t.n * 2 * e.OH + 2 * oy) * (2 * e.OW) + 2 * ox) * 32 + c8 * 4
                         : ((size_t)(t.n * e.OH + oy) * e.OW + ox) * e.Cout + t.n0 + c8 * 4;
      }
#pragma unroll 1
      for (int j = 0; j < NT / 32; ++j) {
        // residual reads do not depend on the accumulator: issue them first, they land under the TMEM load + transpose
        float4 rr[8];
        if (e.res) {
#pragma unroll
          for (int g = 0; g < 8; ++g) rr[g] = ok[g] ? ldg4(e.res + rowoff[g] + j * 32) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float4 bia = make_float4(0.f, 0.f, 0.f, 0.f);
        if (e.bias) bia = ldg4(e.bias + t.n0 + j * 32 + c8 * 4);
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * Cfg::ACC_COLS + j * 32), v);
        if (Cfg::WIDE) {                                         // second column block: 2^11 x the f16(a).r_w correction
          uint32_t u[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * Cfg::ACC_COLS + NT + j * 32), u);
#pragma unroll
          for (int c = 0; c < 32; ++c) v[c] = __float_as_uint(fmaf(__uint_as_float(u[c]), 1.0f / 2048.0f, __uint_as_float(v[c])));
        }
        if (j == NT / 32 - 1) {                                  // accumulator fully read: hand it back to the MMA warp
          tc_fence_before();
          if (CG == 2) mbar_arrive_cluster(mapa_u32(smem_u32(&acc_empty[ab]), 0));
          else         mbar_arrive_local(smem_u32(&acc_empty[ab]));
        }
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4)
          *reinterpret_cast<float4*>(stage + lane * 32 + ((c4 ^ (lane & 7)) << 2)) =
              make_float4(__uint_as_float(v[c4 * 4]), __uint_as_float(v[c4 * 4 + 1]), __uint_as_float(v[c4 * 4 + 2]), __uint_as_float(v[c4 * 4 + 3]));
        __syncwarp();
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const int r = g * 4 + r8;
          float4 o = *reinterpret_cast<const float4*>(stage + r * 32 + ((c8 ^ (r & 7)) << 2));
          o.x += bia.x; o.y += bia.y; o.z += bia.z; o.w += bia.w;
          if (e.res) { o.x += rr[g].x; o.y += rr[g].y; o.z += rr[g].z; o.w += rr[g].w; }
          if (e.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
          // pixel-shuffle store: slab j = (dy, dx) lands on output pixel (2oy + dy, 2ox + dx), 32 channels each
          float* op = e.ps ? e.out + rowoff[g] + ((size_t)(j >> 1) * (2 * e.OW) + (j & 1)) * 32 : e.out + rowoff[g] + j * 32;
          if (ok[g]) st4(op, o);
        }
        __syncwarp();                                            // the staging rows are free for the next slab
      }
    }
    (void)m;
  } else if (X3 && warp >= 7) {                                 // ---------------- splitter (warps 7..10)
    const int tI = threadIdx.x - 224;
    const int nvec = (int)(e.halo_bytes / 16);
    int g = 0;
    for (int tile = w0; tile < e.ntiles; tile += wstep) {
      for (int cq = 0; cq < e.cchunks * NPH; ++cq, ++g) {
        const int hb = g % HB;
        mbar_wait(smem_u32(&halo_full[hb]), (uint32_t)((g / HB) & 1));
        float4* hi = reinterpret_cast<float4*>(base_ptr + (size_t)hb * T2_HALO_STRIDE);
        float4* lo = reinterpret_cast<float4*>(base_ptr + LO0 + (size_t)hb * Cfg::LO_STRIDE);
        if (XM >= 2) {
          // item = (pixel q, pair of adjacent 16-byte chunks): 8 channels.  The TMA wrote chunk c of pixel q at position
          // c ^ (q & 7), so positions (2j, 2j+1) hold the logical chunks (2j ^ r, 2j ^ r ^ 1), r = q & 7: logical 8-channel
          // group j ^ (r >> 1), halves swapped when r is odd.  Each group becomes one 16-byte chunk of the pixel's 64-byte
          // bf16 row, stored at chunk position group ^ ((row address >> 7) & 3)  (SWIZZLE_64B on absolute address bits).
          const uint32_t lo_base = base + LO0 + (uint32_t)hb * Cfg::LO_STRIDE;
          uint8_t* lo_ptr = reinterpret_cast<uint8_t*>(lo);
          for (int i = tI; i < nvec / 2; i += 128) {
            const int q = i >> 2, j = i & 3, r = q & 7;
            // access order within the pair alternates with (thread, row) parity so that the 8 threads of a quarter-warp
            // (two rows) touch 8 different 16-byte bank groups: {0,3,4,7} of the even row, {1,2,5,6} of the odd one
            const int f = (i ^ q) & 1;
            float4 va = hi[q * 8 + 2 * j + f], vb = hi[q * 8 + 2 * j + (f ^ 1)];
            if (XM == 4 || XM == 6) {                          // 16-bit halos: f16(a) (saturating), [XM 4: bf16(a),] bf16(a - f16(a))
              const float4 w0 = f ? vb : va, w1 = f ? va : vb;
              uint4 f16v, a16, r16;
              f16v.x = pack_f16x2_sat(w0.x, w0.y); f16v.y = pack_f16x2_sat(w0.z, w0.w); f16v.z = pack_f16x2_sat(w1.x, w1.y); f16v.w = pack_f16x2_sat(w1.z, w1.w);
              a16.x = pack_bf16x2(w0.x, w0.y); a16.y = pack_bf16x2(w0.z, w0.w); a16.z = pack_bf16x2(w1.x, w1.y); a16.w = pack_bf16x2(w1.z, w1.w);
              r16.x = pack_bf16x2(w0.x - f16_lo(f16v.x), w0.y - f16_hi(f16v.x)); r16.y = pack_bf16x2(w0.z - f16_lo(f16v.y), w0.w - f16_hi(f16v.y));
              r16.z = pack_bf16x2(w1.x - f16_lo(f16v.z), w1.y - f16_hi(f16v.z)); r16.w = pack_bf16x2(w1.z - f16_lo(f16v.w), w1.w - f16_hi(f16v.w));
              if (r & 1) {
                f16v = make_uint4(f16v.z, f16v.w, f16v.x, f16v.y);
                a16 = make_uint4(a16.z, a16.w, a16.x, a16.y);
                r16 = make_uint4(r16.z, r16.w, r16.x, r16.y);
              }
              const uint32_t grp4 = (uint32_t)(j ^ (r >> 1));
#pragma unroll
              for (int tl = 0; tl < (XM == 6 ? 2 : 3); ++tl) {
                const uint32_t row4 = (uint32_t)tl * T2_HALO16_BYTES + (uint32_t)q * 64u;
                *reinterpret_cast<uint4*>(lo_ptr + row4 + ((grp4 ^ (((lo_base + row4) >> 7) & 3u)) << 4)) =
                    tl == 0 ? f16v : ((tl == 1 && XM == 4) ? a16 : r16);
              }
              continue;
            }
            if (XM == 3 || XM == 5) {                          // single-pass 16-bit operands: convert, nothing else
              const float4 w0 = f ? vb : va, w1 = f ? va : vb;
              uint4 a16;
              if (XM == 5) {
                a16.x = pack_f16x2_sat(w0.x, w0.y); a16.y = pack_f16x2_sat(w0.z, w0.w); a16.z = pack_f16x2_sat(w1.x, w1.y); a16.w = pack_f16x2_sat(w1.z, w1.w);
              } else {
                a16.x = pack_bf16x2(w0.x, w0.y); a16.y = pack_bf16x2(w0.z, w0.w); a16.z = pack_bf16x2(w1.x, w1.y); a16.w = pack_bf16x2(w1.z, w1.w);
              }
              if (r & 1) a16 = make_uint4(a16.z, a16.w, a16.x, a16.y);
              const uint32_t grp3 = (uint32_t)(j ^ (r >> 1)), row3 = (uint32_t)q * 64u;
              *reinterpret_cast<uint4*>(lo_ptr + row3 + ((grp3 ^ (((lo_base + row3) >> 7) & 3u)) << 4)) = a16;
              continue;
            }
            const float4 ha = make_float4(tf32_rna(va.x), tf32_rna(va.y), tf32_rna(va.z), tf32_rna(va.w));
            const float4 hb = make_float4(tf32_rna(vb.x), tf32_rna(vb.y), tf32_rna(vb.z), tf32_rna(vb.w));
            hi[q * 8 + 2 * j + f] = ha;
            hi[q * 8 + 2 * j + (f ^ 1)] = hb;
            const float4 v0 = f ? vb : va, v1 = f ? va : vb, h0 = f ? hb : ha, h1 = f ? ha : hb;
            uint4 a16, l16;                                   // bf16(a), bf16(a - tf32(a)) in position order
            a16.x = pack_bf16x2(v0.x, v0.y); a16.y = pack_bf16x2(v0.z, v0.w); a16.z = pack_bf16x2(v1.x, v1.y); a16.w = pack_bf16x2(v1.z, v1.w);
            l16.x = pack_bf16x2(v0.x - h0.x, v0.y - h0.y); l16.y = pack_bf16x2(v0.z - h0.z, v0.w - h0.w);
            l16.z = pack_bf16x2(v1.x - h1.x, v1.y - h1.y); l16.w = pack_bf16x2(v1.z - h1.z, v1.w - h1.w);
            if (r & 1) {                                      // position 2j holds the ODD logical chunk: swap the halves
              a16 = make_uint4(a16.z, a16.w, a16.x, a16.y);
              l16 = make_uint4(l16.z, l16.w, l16.x, l16.y);
            }
            const uint32_t grp = (uint32_t)(j ^ (r >> 1));
            const uint32_t row_hi = (uint32_t)q * 64u, row_lo = T2_HALO16_BYTES + (uint32_t)q * 64u;
            const uint32_t off_hi = row_hi + ((grp ^ (((lo_base + row_hi) >> 7) & 3u)) << 4);
            const uint32_t off_lo = row_lo + ((grp ^ (((lo_base + row_lo) >> 7) & 3u)) << 4);
            *reinterpret_cast<uint4*>(lo_ptr + off_hi) = a16;
            *reinterpret_cast<uint4*>(lo_ptr + off_lo) = l16;
          }
        } else
        for (int i = tI; i < nvec; i += 128) {
          const float4 v = hi[i];
          const float4 h = make_float4(tf32_rna(v.x), tf32_rna(v.y), tf32_rna(v.z), tf32_rna(v.w));
          hi[i] = h;
          lo[i] = make_float4(tf32_rna(v.x - h.x), tf32_rna(v.y - h.y), tf32_rna(v.z - h.z), tf32_rna(v.w - h.w));
        }
        fence_async_smem();
        if (CG == 2) mbar_arrive_cluster(mapa_u32(smem_u32(&halo_ready[hb]), 0));
        else         mbar_arrive_local(smem_u32(&halo_ready[hb]));
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
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode2() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  });
  return fn;
}
struct Key2 {
  const void* ptr; int d0, d1, d2, d3, b1, b2;   // b2 also encodes element stride / bf16 (see get_map2)
  bool operator==(const Key2& o) const { return ptr == o.ptr && d0 == o.d0 && d1 == o.d1 && d2 == o.d2 && d3 == o.d3 && b1 == o.b1 && b2 == o.b2; }
};
struct Key2Hash {
  size_t operator()(const Key2& k) const {
    size_t h = (size_t)k.ptr;
    for (int v : {k.d0, k.d1, k.d2, k.d3, k.b1, k.b2}) h = h * 1000003u ^ (size_t)v;
    return h;
  }
};
std::mutex g_mu2;
std::unordered_map<Key2, CUtensorMap, Key2Hash> g_maps2;

// b1, b2: box extent in ELEMENTS FETCHED along dims 1, 2; es = element stride along those dims (1 or 2)
// bf16 = true: a [d1][d0] bf16 matrix read in {32, b1} boxes with SWIZZLE_64B (the filter's bf16 hi / lo images)
int get_map2(CUtensorMap* out, const void* ptr, int rank, int d0, int d1, int d2, int d3, int b1, int b2, int es = 1,
             bool bf16 = false) {
  Key2 key{ptr, d0, d1, d2, d3, b1 * es, b2 * es + (es - 1) + (bf16 ? 1000 : 0)};
  {
    std::lock_guard<std::mutex> lk(g_mu2);
    auto it = g_maps2.find(key);
    if (it != g_maps2.end()) { *out = it->second; return 0; }
  }
  EncodeTiledFn enc = get_encode2();
  if (!enc) return DH_E_VARIANT;
  cuuint64_t dims[4] = {(cuuint64_t)d0, (cuuint64_t)d1, (cuuint64_t)d2, (cuuint64_t)d3};
  const cuuint64_t esz = bf16 ? 2 : 4;
  cuuint64_t strides[3] = {(cuuint64_t)d0 * esz, (cuuint64_t)d0 * d1 * esz, (cuuint64_t)d0 * d1 * d2 * esz};
  cuuint32_t box[4] = {32, (cuuint32_t)(b1 * es), (cuuint32_t)(b2 * es), 1};
  cuuint32_t estr[4] = {1, (cuuint32_t)es, (cuuint32_t)es, 1};
  CUtensorMap m;
  const CUresult r = enc(&m, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank,
                         (void*)ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         bf16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return DH_E_SHAPE;
  {
    std::lock_guard<std::mutex> lk(g_mu2);
    if (g_maps2.size() > 4096) g_maps2.clear();
    g_maps2[key] = m;
  }
  *out = m;
  return 0;
}

}  // namespace

// generic fp32 tiled tensor map (used by the stem for its planar NCHW halo); strides in bytes for dims 1..rank-1
int dh_encode_tiled_f32(CUtensorMap* out, const void* ptr, int rank, const unsigned long long* dims,
                        const unsigned long long* strides, const unsigned* box, bool swizzle128) {
  return dh_encode_tiled_f32_sw(out, ptr, rank, dims, strides, box, swizzle128 ? 128 : 0);
}
// swizzle_bytes: 0 (none), 64 or 128
static int encode_tiled_sw(CUtensorMapDataType dtype, CUtensorMap* out, const void* ptr, int rank, const unsigned long long* dims,
                           const unsigned long long* strides, const unsigned* box, int swizzle_bytes) {
  EncodeTiledFn enc = get_encode2();
  if (!enc) return DH_E_VARIANT;
  cuuint64_t d[5], st[4];
  cuuint32_t b[5], es[5] = {1, 1, 1, 1, 1};
  for (int i = 0; i < rank; ++i) { d[i] = dims[i]; b[i] = box[i]; }
  for (int i = 0; i + 1 < rank; ++i) st[i] = strides[i];
  const CUresult r = enc(out, dtype, (cuuint32_t)rank, const_cast<void*>(ptr), d, st, b, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE,
                         swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE),
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : DH_E_SHAPE;
}
int dh_encode_tiled_f32_sw(CUtensorMap* out, const void* ptr, int rank, const unsigned long long* dims,
                           const unsigned long long* strides, const unsigned* box, int swizzle_bytes) {
  return encode_tiled_sw(CU_TENSOR_MAP_DATA_TYPE_FLOAT32, out, ptr, rank, dims, strides, box, swizzle_bytes);
}
int dh_encode_tiled_f16_sw(CUtensorMap* out, const void* ptr, int rank, const unsigned long long* dims,
                           const unsigned long long* strides, const unsigned* box, int swizzle_bytes) {
  return encode_tiled_sw(CU_TENSOR_MAP_DATA_TYPE_FLOAT16, out, ptr, rank, dims, strides, box, swizzle_bytes);
}

namespace {
template <int NT, int XM, int KS, int SD, int CG>
int launch2k(const CUtensorMap& A0, const CUtensorMap& A1, const CUtensorMap& Bm, const CUtensorMap& B16, const CUtensorMap& B16f, const T2Args& e, dim3 grid,
             cudaStream_t s) {
  using Cfg = T2Cfg<NT, XM, CG>;
  auto kern = conv_tc2_kernel<NT, XM, KS, SD, CG>;
  cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
  if (err != cudaSuccess) return (int)err;
  if (CG == 1) {
    kern<<<grid, Cfg::THREADS, Cfg::SMEM, s>>>(A0, A1, Bm, B16, B16f, e);
  } else {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = dim3(Cfg::THREADS, 1, 1); cfg.dynamicSmemBytes = Cfg::SMEM; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    err = cudaLaunchKernelEx(&cfg, kern, A0, A1, Bm, B16, B16f, e);
    if (err != cudaSuccess) return (int)err;
  }
  DH_CHECK_LAUNCH();
  return 0;
}
template <int NT, int XM, int CG>
int launch2(const CUtensorMap& A0, const CUtensorMap& A1, const CUtensorMap& Bm, const CUtensorMap& B16, const CUtensorMap& B16f, const T2Args& e, dim3 grid,
            cudaStream_t s) {
  if (e.stride == 2)
    return e.ntaps == 9 ? launch2k<NT, XM, 3, 2, CG>(A0, A1, Bm, B16, B16f, e, grid, s) : launch2k<NT, XM, 1, 2, CG>(A0, A1, Bm, B16, B16f, e, grid, s);
  return e.ntaps == 9 ? launch2k<NT, XM, 3, 1, CG>(A0, A1, Bm, B16, B16f, e, grid, s) : launch2k<NT, XM, 1, 1, CG>(A0, A1, Bm, B16, B16f, e, grid, s);
}
template <int XM, int CG>
int launch2n(int NT, const CUtensorMap& A0, const CUtensorMap& A1, const CUtensorMap& Bm, const CUtensorMap& B16, const CUtensorMap& B16f, const T2Args& e,
             dim3 grid, cudaStream_t s) {
  switch (NT) {
    case 128: return launch2<128, XM, CG>(A0, A1, Bm, B16, B16f, e, grid, s);
    case 64: return launch2<64, XM, CG>(A0, A1, Bm, B16, B16f, e, grid, s);
    default: return launch2<32, XM, CG>(A0, A1, Bm, B16, B16f, e, grid, s);
  }
}
}  // namespace

bool dh_conv_tc2_eligible(const ConvArgs& a) {
  const bool base = a.wt != nullptr && a.up == 1 &&
                    (a.stride == 1 || (a.stride == 2 && a.inH % 2 == 0 && a.inW % 2 == 0 && !a.ps)) && a.KH == a.KW && (a.KH == 1 || a.KH == 3) &&
                    a.pad == a.KH / 2 && a.C0 > 0 && a.C0 % 32 == 0 && a.C1 % 32 == 0 &&
                    (a.Cout == 32 || a.Cout == 64 || a.Cout == 128 || a.Cout == 256) && a.inH >= 1 && a.inW >= 1;
  if (!base) return false;
  if (a.ps) return a.Cout == 128 && a.res == nullptr;
  return true;
}

// a.wt: [2][Cout][K] = TF32-rounded filter (hi) followed by its TF32-rounded remainder (lo); x3 uses both.
// xm = 6: xm = 4 with the f16(a).r_w correction folded into the main MMA (fifth plane of a.wt: f16(2^11 (w - f16(w)))).
// xm = 5: single-pass f16 operands (saturating; TF32-grade significand at bf16-mode cost).
// xm = 4: f16 main product + bf16 corrections (a.wt then carries a fourth plane: f16(w) | bf16(w - f16(w))).
// xm: 0 = 1xTF32, 1 = 3xTF32 (three TF32 MMAs), 2 = 3xTF32 with the two correction products in bf16, 3 = bf16 operands only.
// cg = 2: CTA pairs (tcgen05 cta_group::2): M = 256 per MMA, each CTA loads and reads only half of the filter tile
// a.wt: [hi fp32 Cout*K][lo fp32 Cout*K][bf16(w) Cout*K][bf16(w - hi) Cout*K]  (engine.kmajor_split)
int dh_launch_conv_tc2(const ConvArgs& a, int xm, int cg, cudaStream_t s) {
  DH_REQUIRE(a.in0 && a.wt && a.out, DH_E_NULL);
  DH_REQUIRE(a.C1 == 0 || a.in1, DH_E_NULL);
  DH_REQUIRE(dh_conv_tc2_eligible(a), DH_E_SHAPE);
  DH_REQUIRE(dh_aligned16(a.in0) && dh_aligned16(a.in1) && dh_aligned16(a.wt) && dh_aligned16(a.out) &&
             dh_aligned16(a.bias) && dh_aligned16(a.res), DH_E_ALIGN);
  const int Cin = a.C0 + a.C1, K = a.KH * a.KW * Cin;
  const int NT = a.Cout >= 128 ? 128 : a.Cout;
  const int hw = (a.KH == 3) ? T2_HW : T2_TW, hh = (a.KH == 3) ? T2_HH : T2_TH;
  CUtensorMap A0, A1, Bm;
  int rc = get_map2(&A0, a.in0, 4, a.C0, a.inW, a.inH, a.N, hw, hh, a.stride);
  if (rc) return rc;
  if (a.C1) { rc = get_map2(&A1, a.in1, 4, a.C1, a.inW, a.inH, a.N, hw, hh, a.stride); if (rc) return rc; } else A1 = A0;
  cg = (cg == 2 && xm < 3) ? 2 : 1;
  rc = get_map2(&Bm, a.wt, 2, K, 2 * a.Cout, 1, 1, NT / cg, 1);  // rows [0,Cout) = hi, [Cout,2Cout) = lo
  if (rc) return rc;
  CUtensorMap B16 = Bm;
  if (xm >= 2) {                                                 // bf16 images follow the two fp32 ones
    rc = get_map2(&B16, a.wt + (size_t)2 * a.Cout * K, 2, K, 2 * a.Cout, 1, 1, NT / cg, 1, 1, true);
    if (rc) return rc;
  }
  CUtensorMap B16f = B16;
  if (xm >= 4) {                                                 // fourth plane: f16(w) | bf16(w - f16(w))
    rc = get_map2(&B16f, a.wt + (size_t)3 * a.Cout * K, 2, K, 2 * a.Cout, 1, 1, NT, 1, 1, true);
    if (rc) return rc;
  }
  if (xm == 6) {                                                 // fifth plane: f16(2^11 (w - f16(w))); rides in the fp32 map's slot
    rc = get_map2(&Bm, a.wt + (size_t)4 * a.Cout * K, 2, K, 2 * a.Cout, 1, 1, NT, 1, 1, true);
    if (rc) return rc;
  }
  T2Args e;
  e.bias = a.bias; e.res = a.res; e.out = a.out;
  e.OH = a.inH / a.stride; e.OW = a.inW / a.stride; e.Cout = a.Cout; e.relu = a.relu; e.stride = a.stride;
  e.tilesX = dh_cdiv(e.OW, T2_TW);
  e.cchunks0 = a.C0 / 32; e.cchunks = Cin / 32; e.ntaps = a.KH * a.KW; e.KW = a.KW; e.Cin = Cin; e.ps = a.ps;
  e.halo_w = hw; e.halo_h = hh; e.halo_bytes = (uint32_t)(hw * hh * 128);
  e.tilesY = dh_cdiv(e.OH, T2_TH); e.ncout_tiles = a.Cout / NT;
  e.N = a.N;
  const int mtiles = e.tilesX * e.tilesY * a.N;
  e.ntiles = (cg == 2 ? (mtiles + 1) / 2 : mtiles) * e.ncout_tiles;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (cg == 2) {
    const int pairs = sms / 2;
    dim3 grid((unsigned)(2 * (e.ntiles < pairs ? e.ntiles : pairs)), 1, 1);       // persistent: one CTA pair per TPC
    if (xm == 2) return launch2n<2, 2>(NT, A0, A1, Bm, B16, B16f, e, grid, s);
    return xm ? launch2n<1, 2>(NT, A0, A1, Bm, B16, B16f, e, grid, s) : launch2n<0, 2>(NT, A0, A1, Bm, B16, B16f, e, grid, s);
  }
  dim3 grid((unsigned)((e.ntiles < sms || a.flat) ? e.ntiles : sms), 1, 1);   // persistent: one CTA per SM (flat: one per tile)
  if (xm == 6) return launch2n<6, 1>(NT, A0, A1, Bm, B16, B16f, e, grid, s);
  if (xm == 5) return launch2n<5, 1>(NT, A0, A1, Bm, B16, B16f, e, grid, s);
  if (xm == 4) return launch2n<4, 1>(NT, A0, A1, Bm, B16, B16f, e, grid, s);
  if (xm == 3) return launch2n<3, 1>(NT, A0, A1, Bm, B16, B16f, e, grid, s);
  if (xm == 2) return launch2n<2, 1>(NT, A0, A1, Bm, B16, B16f, e, grid, s);
  return xm ? launch2n<1, 1>(NT, A0, A1, Bm, B16, B16f, e, grid, s) : launch2n<0, 1>(NT, A0, A1, Bm, B16, B16f, e, grid, s);
}
